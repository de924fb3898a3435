// greedy_host.cpp -- TEST HARNESS ONLY (never loaded by the product package).
// Compiles the greedy agent of azb_rules.cuh -- greedy_action and opponent_greedy, the code the CUDA kernels include -- with
// g++, so that it can be compared with the naive restatement (greedy_oracle.c) on the CPU.  Works on unpacked records.
#include <cstdint>
#include "../../azul_deep_reinforcement_learning_b200/csrc/azb_rules.cuh"

using namespace azb;

template <int P, int POOL>
static int run_greedy_action(const int32_t* rec, uint32_t word)
{
    Game<P> g;
    if (!import_record<P>(g, [&](int i) { return rec[i]; })) return -16;
    uint32_t m[6];
    legal_mask(g, m);
    return (int)greedy_action<P, POOL>(g, m, word);
}

template <int P, int POOL>
static int run_opponent_greedy(int32_t* rec, uint64_t seed, uint32_t gid, int require_two, uint32_t* mask6, int32_t* diff)
{
    Game<P> g;
    if (!import_record<P>(g, [&](int i) { return rec[i]; })) return -16;
    Philox rng{(uint32_t)seed, (uint32_t)(seed >> 32)};
    *diff = opponent_greedy<P, POOL>(g, rng, gid, require_two != 0, mask6);
    export_record<P>(g, [&](int i, int32_t v) { rec[i] = v; });
    return 0;
}

#define GH_DISPATCH(CALL, ARGS)                                                                                \
    if (players == 2 && pool == 0) return CALL<2, 0> ARGS; if (players == 2 && pool == 1) return CALL<2, 1> ARGS;   \
    if (players == 3 && pool == 0) return CALL<3, 0> ARGS; if (players == 3 && pool == 1) return CALL<3, 1> ARGS;   \
    if (players == 4 && pool == 0) return CALL<4, 0> ARGS; if (players == 4 && pool == 1) return CALL<4, 1> ARGS;   \
    return -101;

// the action (180: none legal), or -16 for a record that cannot be packed
extern "C" int hh_greedy_action(const int32_t* rec, int players, int pool, uint32_t word)
{
    GH_DISPATCH(run_greedy_action, (rec, word))
}

extern "C" int hh_opponent_greedy(int32_t* rec, int players, int pool, uint64_t seed, uint32_t gid, int require_two,
                                  uint32_t* mask6, int32_t* diff)
{
    GH_DISPATCH(run_opponent_greedy, (rec, seed, gid, require_two, mask6, diff))
}
