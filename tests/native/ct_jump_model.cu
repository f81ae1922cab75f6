// Host-only model of phase 4 of ct_build_kernel (cs267_hw3_b200/csrc/ctable.cuh): the pointer jumping in shared memory
// that tells every node of a chunk its segment head and its distance from it.  Built with nvcc against the shipped
// header (runs without a GPU), so it uses the shipped kCtBuildThreads, KH_CT_JUMPS, CtBuild<W>::kMaxSlots and
// CtBuild<W>::kJumpRounds.
//
// The loop structure is the kernel's: thread t owns nodes t, t + T, t + 2T, ... and keeps a bit per unsettled node;
// a round is KH_CT_JUMPS in-place passes over those nodes, then a barrier that ends the loop when no thread has an
// unsettled node left.  The schedule is the one the memory model allows and that is worst for progress: a thread
// sees its own writes at once, and every other thread's node as it stood at the last barrier.
//
// The chunk is one chain of L nodes whose ids are randomly permuted (the staging atomics hand out record positions in
// no particular order): a head, then L - 1 nodes that each point at their predecessor at distance 1.
//
//   ct_jump_model W L seed
// prints one line:
//   J threads max_slots cap  rounds_run unsettled_at_cap  rounds_to_settle
// rounds_run / unsettled_at_cap: the shipped loop (cap = CtBuild<W>::kJumpRounds rounds); a node counts as unsettled
// if its ancestor is not the head or its distance is not its place in the chain.  rounds_to_settle: the same schedule
// without a cap, the first barrier after which every node is settled.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "../../cs267_hw3_b200/csrc/ctable.cuh"

using namespace kh;

struct Run {
    int rounds_run = 0, rounds_to_settle = -1;
    u32 unsettled = 0;
};

static u32 count_unsettled(const std::vector<u32>& pd, const std::vector<u32>& pos) {
    u32 bad = 0;
    for (u32 node = 0; node < pd.size(); ++node) {
        const u32 a = pd[node] >> 16;
        if (a == node) continue;                                           // the head
        const bool root = (pd[a] >> 16) == a;
        if (!root || (pd[node] & 0xFFFFu) != pos[node]) ++bad;
    }
    return bad;
}

static Run run(u32 L, u64 seed, int cap) {
    const u32 T = (u32)kCtBuildThreads;
    std::vector<u32> perm(L), pos(L), pd(L);
    for (u32 i = 0; i < L; ++i) perm[i] = i;
    std::mt19937_64 rng(seed);
    std::shuffle(perm.begin(), perm.end(), rng);
    for (u32 p = 0; p < L; ++p) {
        const u32 node = perm[p];
        pos[node] = p;
        pd[node] = p == 0 ? (node << 16) : ((perm[p - 1] << 16) | 1u);   // head: (itself, segment index 0)
    }
    std::vector<u32> active(T, 0);
    for (u32 t = 0; t < T; ++t)
        for (u32 i = 0, node = t; node < L; ++i, node += T) active[t] |= ((pd[node] >> 16) != node) ? (1u << i) : 0u;
    Run r;
    std::vector<u32> snap;
    for (int round = 0; round < cap; ++round) {
        snap = pd;                                                         // what every thread sees of the others this round
        for (u32 t = 0; t < T; ++t) {
            for (int rep = 0; rep < KH_CT_JUMPS; ++rep) {
                for (u32 m = active[t]; m; m &= m - 1u) {
                    const u32 i = (u32)__builtin_ctz(m), node = t + i * T;
                    const u32 pdv = pd[node], a = pdv >> 16;
                    const u32 pa = (a % T == t) ? pd[a] : snap[a], a2 = pa >> 16;
                    if (a2 == a) { active[t] &= ~(1u << i); continue; }
                    pd[node] = (a2 << 16) | ((pdv + pa) & 0xFFFFu);
                }
            }
        }
        r.rounds_run = round + 1;
        if (r.rounds_to_settle < 0 && count_unsettled(pd, pos) == 0) r.rounds_to_settle = round + 1;
        bool any = false;
        for (u32 t = 0; t < T; ++t) any |= active[t] != 0;
        if (!any) break;
    }
    r.unsettled = count_unsettled(pd, pos);
    return r;
}

template <int W>
static int main_w(u32 L, u64 seed) {
    typedef CtBuild<W> B;
    if (L < 1 || L > B::kMaxSlots) { fprintf(stderr, "L must be in [1, %u]\n", B::kMaxSlots); return 2; }
    const Run shipped = run(L, seed, B::kJumpRounds);
    const Run open = run(L, seed, 64);
    printf("%d %d %u %d  %d %u  %d\n", KH_CT_JUMPS, kCtBuildThreads, B::kMaxSlots, B::kJumpRounds, shipped.rounds_run,
           shipped.unsettled, open.rounds_to_settle);
    return 0;
}

int main(int argc, char** argv) {
    if (argc != 4) { fprintf(stderr, "usage: ct_jump_model W L seed\n"); return 2; }
    const int W = atoi(argv[1]);
    const u32 L = (u32)strtoul(argv[2], nullptr, 10);
    const u64 seed = strtoull(argv[3], nullptr, 10);
    if (W == 1) return main_w<1>(L, seed);
    if (W == 2) return main_w<2>(L, seed);
    fprintf(stderr, "W must be 1 or 2\n");
    return 2;
}
