// Host-only harness over the product's LIKE pattern classifier (plan_b200/csrc/plan_ir.hpp like_segments): reads one
// hex-encoded pattern per line ('-' is the empty pattern), prints "1 <seg hex>,<seg hex>,..." when the pattern runs as
// segment-by-segment word search, "0" otherwise.  tests/test_like_segments_cpu.py checks the answers.
#include <stdio.h>

#include <iostream>
#include <string>
#include <vector>

#include "../../plan_b200/csrc/plan_ir.hpp"

using namespace pg;

int main()
{
    std::string hex;
    while (std::cin >> hex) {
        std::string pat;
        if (hex != "-")
            for (size_t i = 0; i + 1 < hex.size(); i += 2) pat += (char)std::stoi(hex.substr(i, 2), nullptr, 16);
        std::vector<std::string> segs;
        if (!like_segments(pat, &segs)) { printf("0\n"); continue; }
        printf("1 ");
        for (size_t s = 0; s < segs.size(); s++) {
            if (s) printf(",");
            for (unsigned char ch : segs[s]) printf("%02x", ch);
        }
        printf("\n");
    }
    return 0;
}
