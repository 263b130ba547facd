"""The LIKE pattern classifier of the grouped LEFT-join count (plan_ir.hpp like_segments), run on the host by
tests/hostlogic/likeseg_check.cu -- no GPU.  A pattern `%s1%...%sk%` (1 <= k <= 4 segments of 1..8 bytes, no '_', runs of '%'
taken as one) runs as k word-at-a-time searches, each starting where the previous match ended; everything else takes the
byte-wise wildcardMatch.  Also pins why that is exact: for such patterns, greedy leftmost segment search gives what
wildcardMatch gives."""
import os
import random
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _expected(pat):
    """restatement of the rule: (qualifies, segments)"""
    if len(pat) < 3 or pat[:1] != b"%" or pat[-1:] != b"%" or b"_" in pat:
        return False, []
    segs = [s for s in pat.split(b"%") if s]
    if not 1 <= len(segs) <= 4 or any(len(s) > 8 for s in segs):
        return False, []
    return True, segs


def _greedy(segs, target):
    pos = 0
    for s in segs:
        i = target.find(s, pos)
        if i < 0:
            return False
        pos = i + len(s)
    return True


def _classify(tmp_path, pats):
    exe = str(tmp_path / "likeseg_check")
    src = os.path.join(ROOT, "tests", "hostlogic", "likeseg_check.cu")
    subprocess.run(["/usr/local/cuda/bin/nvcc", "-std=c++17", "-O1", "-Wno-deprecated-gpu-targets", "-o", exe, src], check=True, capture_output=True)
    inp = "".join((p.hex() or "-") + "\n" for p in pats)
    out = subprocess.run([exe], input=inp, capture_output=True, text=True, check=True).stdout.split("\n")
    got = []
    for line in out[:len(pats)]:
        if line == "0":
            got.append((False, []))
        else:
            flag, segs = line.split(" ")
            assert flag == "1"
            got.append((True, [bytes.fromhex(s) for s in segs.split(",")]))
    return got


LISTED = [
    (b"%pending%accounts%", [b"pending", b"accounts"]),
    (b"%special%requests%", [b"special", b"requests"]),
    (b"%ly%final%ironic%", [b"ly", b"final", b"ironic"]),
    (b"%%pending%%accounts%%", [b"pending", b"accounts"]),
    (b"%accounts%", [b"accounts"]),
    (b"%a%b%c%d%", [b"a", b"b", b"c", b"d"]),
    (b"%%%x%%%", [b"x"]),
    (b"%\x80\xff%", [b"\x80\xff"]),
    (b"%furiously%", None),                # a 9-byte segment
    (b"%pend_ng%accounts%", None),         # '_'
    (b"pending%accounts%", None),          # no leading '%'
    (b"%pending%accounts", None),          # no trailing '%'
    (b"%a%b%c%d%e%", None),                # five segments
    (b"%%", None), (b"%", None), (b"", None), (b"%%%", None), (b"abc", None),
]


def test_like_segments_classifies_listed_and_random_patterns(tmp_path):
    rng = random.Random(13)
    pats = [p for p, _ in LISTED]
    alphabet = b"ab%_xy\x80"
    for _ in range(3000):
        pats.append(bytes(rng.choice(alphabet) for _ in range(rng.randrange(0, 24))))
    for _ in range(1000):      # mostly well-formed: '%' around 1..5 segments of 1..10 bytes, runs of '%'
        segs = [bytes(rng.choice(b"abcxyz\x90") for _ in range(rng.randrange(1, 11))) for _ in range(rng.randrange(1, 6))]
        pats.append(b"%" * rng.randrange(1, 3) + b"".join(s + b"%" * rng.randrange(1, 3) for s in segs))
    got = _classify(tmp_path, pats)
    for (p, want), g in zip(LISTED, got):
        assert g == ((want is not None), want or []), (p, g)
    for p, g in zip(pats, got):
        assert g == _expected(p), (p, g)
    assert sum(1 for g in got if g[0]) > 400


def test_greedy_segment_search_is_wildcard_match():
    """the device's segment-by-segment search restated: equal to wildcardMatch on qualifying patterns over random and
    adversarial targets (overlapping candidates, the second word only before the first, empty and short strings)"""
    from oracle import oracle as O
    rng = random.Random(29)
    cases = [(b"%pending%accounts%", t) for t in (b"", b"pend", b"accounts pending", b"pendpendingaccounts", b"pendingaccounts",
                                                   b"xx pending yy accounts", b"pending accounts\x80")]
    cases += [(b"%ly%ly%", t) for t in (b"ly", b"lyly", b"lly", b"l y ly", b"")]
    for _ in range(5000):
        segs = [bytes(rng.choice(b"ab") for _ in range(rng.randrange(1, 4))) for _ in range(rng.randrange(1, 5))]
        pat = b"%" + b"%".join(segs) + b"%"
        cases.append((pat, bytes(rng.choice(b"ab\x80") for _ in range(rng.randrange(0, 16)))))
    for pat, t in cases:
        ok, segs = _expected(pat)
        assert ok
        assert _greedy(segs, t) == O.wildcard_match(pat, t), (pat, t)
