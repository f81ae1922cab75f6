// Host check of ct_jump_link (cs267_hw3_b200/csrc/ctable.cuh), the per-link update of ct_rank_round_kernel: the
// pointer-jumping fallback of a chunk-table traverse.  Built with nvcc against the shipped header (runs without a GPU),
// so it uses the shipped function and kCtMaxRounds.
//
// A segment list is a link per segment: (successor << 32) | characters of the segment, or (kLinkTail << 32) for the
// last one.  The rounds are lockstep: every link of a round reads the others as they stood after the previous round.
//
//   ct_link_jump_check cycle   a head stub (distance 0) in front of a cycle of L segments whose lengths average
//                              1 .. 6000 characters; after kCtMaxRounds rounds no link of it may be final (a final
//                              head stub would make the traverse claim a segment of the cycle as its contig's tail)
//   ct_link_jump_check chain   chains of L segments: after enough rounds every link is final, points at the last
//                              segment and holds the exact number of characters up to it
// Prints "ok <cases>" and exits 0, or prints the first failure and exits 1.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "../../cs267_hw3_b200/csrc/ctable.cuh"

using namespace kh;

static u64 open_link(u32 to, u32 chars) { return ((u64)to << 32) | chars; }

// the rounds of ct_rank_round_kernel over one list; returns the number of rounds in which some link jumped
static int run_rounds(std::vector<u64>& link, int rounds) {
    int moved = 0;
    std::vector<u64> snap;
    for (int r = 0; r < rounds; ++r) {
        snap = link;
        bool any = false;
        for (size_t i = 0; i < link.size(); ++i) {
            const u64 li = snap[i];
            const u32 pi = (u32)(li >> 32);
            if (pi >= kLinkCtFirstMarker || ((u32)li & kLinkFinalBit)) continue;
            const u64 lp = snap[pi];
            link[i] = ct_jump_link(li, lp);
            any |= link[i] != li && (u32)(lp >> 32) < kLinkCtFirstMarker;
        }
        if (!any) break;
        ++moved;
    }
    return moved;
}

// segment lengths of mean `avg` (1 .. 2 avg - 1, each below the 24-bit meta field)
static std::vector<u32> lengths(u32 n, u32 avg, std::mt19937_64& rng) {
    std::vector<u32> len(n);
    std::uniform_int_distribution<u32> d(1, 2 * avg - 1);
    for (auto& v : len) v = d(rng);
    return len;
}

static int check_cycles() {
    const u32 sizes[] = {1, 2, 3, 5, 64, 1000};
    u64 cases = 0;
    std::mt19937_64 rng(1);
    for (u32 L : sizes) {
        for (u32 avg = 1; avg <= 6000; ++avg) {
            // link 0: the head stub of a start node (no characters), links 1 .. L: the cycle
            const std::vector<u32> len = lengths(L, avg, rng);
            std::vector<u64> link(L + 1);
            link[0] = open_link(1, 0);
            for (u32 j = 0; j < L; ++j) link[1 + j] = open_link(1 + (j + 1) % L, len[j]);
            run_rounds(link, kCtMaxRounds);
            for (u32 i = 0; i <= L; ++i) {
                if ((u32)link[i] & kLinkFinalBit) {
                    printf("cycle L=%u avg=%u: link %u (%s) is final after %d rounds: distance word 0x%08x\n", L, avg, i,
                           i ? "cycle" : "head stub", kCtMaxRounds, (u32)link[i]);
                    return 1;
                }
            }
            ++cases;
        }
    }
    printf("ok %llu\n", (unsigned long long)cases);
    return 0;
}

static int check_chains() {
    struct Case { u32 L, avg; };
    // avg 0: every segment 2^24 - 1 characters (the most a meta word holds); with 129 segments the head stub's
    // distance is 2^31 - 128, just under the limit
    const Case cases[] = {{1, 5}, {2, 1}, {3, 7}, {17, 40}, {1000, 100}, {4097, 3}, {1u << 20, 2}, {127, 1u << 23}, {129, 0}};
    u64 n = 0;
    std::mt19937_64 rng(2);
    for (const Case& c : cases) {
        std::vector<u32> len = c.avg ? lengths(c.L, c.avg, rng) : std::vector<u32>(c.L, 0xFFFFFFu);
        for (auto& v : len) v = v > 0xFFFFFFu ? 0xFFFFFFu : v;
        // link 0: head stub; links 1 .. L: the chain; link L is the last segment (its characters live in meta)
        std::vector<u64> link(c.L + 1);
        link[0] = open_link(1, 0);
        for (u32 j = 1; j < c.L; ++j) link[j] = open_link(j + 1, len[j - 1]);
        link[c.L] = (u64)kLinkTail << 32;
        std::vector<u64> dist(c.L + 1, 0);               // characters from segment j to the last one
        for (u32 j = c.L - 1; j >= 1; --j) dist[j] = dist[j + 1] + len[j - 1];
        dist[0] = dist[1];
        if (dist[0] >= kLinkDistMask) { printf("chain L=%u: test case too long\n", c.L); return 1; }
        const int moved = run_rounds(link, kCtMaxRounds);
        int need = 0;
        while ((1ull << need) < c.L) ++need;             // a stub + L segments: ceil(log2 L) rounds of jumps
        if (moved > need) { printf("chain L=%u: %d rounds moved, at most %d expected\n", c.L, moved, need); return 1; }
        for (u32 j = 0; j < c.L; ++j) {
            const u64 want = ((u64)c.L << 32) | kLinkFinalBit | (u32)dist[j];
            if (link[j] != want) {
                printf("chain L=%u: link %u is 0x%016llx, expected 0x%016llx\n", c.L, j, (unsigned long long)link[j],
                       (unsigned long long)want);
                return 1;
            }
        }
        if (link[c.L] != ((u64)kLinkTail << 32)) { printf("chain L=%u: the last segment's link changed\n", c.L); return 1; }
        ++n;
    }
    // the targets the update leaves alone or closes: pending / unused successors, and every end marker
    const u64 li = open_link(7, 12);
    for (u32 m : {kLinkPending, kLinkUnused})
        if (ct_jump_link(li, (u64)m << 32) != li) { printf("marker 0x%08x: an open link changed\n", m); return 1; }
    for (u32 m : {kLinkTail, kLinkClaimed, kLinkMissing, kLinkConverge})
        if (ct_jump_link(li, (u64)m << 32) != (li | kLinkFinalBit)) { printf("marker 0x%08x: the link did not turn final\n", m); return 1; }
    // saturation: a sum at or past the distance limit stays open, whatever the target's final bit says
    if (ct_jump_link(open_link(3, kLinkDistMask - 5), open_link(4, 5) | kLinkFinalBit) != open_link(4, kLinkDistMask) ||
        ct_jump_link(open_link(3, kLinkDistMask), open_link(4, kLinkDistMask)) != open_link(4, kLinkDistMask) ||
        ct_jump_link(open_link(3, kLinkDistMask - 6), open_link(4, 5) | kLinkFinalBit) != (open_link(4, kLinkDistMask - 1) | kLinkFinalBit)) {
        printf("saturation at the distance limit is wrong\n");
        return 1;
    }
    printf("ok %llu\n", (unsigned long long)n);
    return 0;
}

int main(int argc, char** argv) {
    if (argc == 2 && !strcmp(argv[1], "cycle")) return check_cycles();
    if (argc == 2 && !strcmp(argv[1], "chain")) return check_chains();
    fprintf(stderr, "usage: ct_link_jump_check cycle|chain\n");
    return 2;
}
