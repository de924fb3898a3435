// azb_rules.cuh -- the Azul rules on the bit-packed game state, one game per thread.
//
// Everything here is new code written for the packed layout below; the behaviour it must
// reproduce is the reference's azulnet/azul.py (cited per function).  The functions are
// __host__ __device__ so that tests/harness can compile the very same header with g++ and
// compare it with the oracle on the CPU before any GPU time is spent; the product only ever
// calls them from the kernels in azb_kernels.cu.
//
// Packed state, W(P) = 7 + 5*P uint32 words per game, stored structure-of-arrays in HBM
// (word w of game g at state[w * stride + g], so a warp reads 32 consecutive words):
//
//   shared words
//   0..2  PL0, PL1, PL2  bit-planes of the 30 (source, colour) tile counts: bit (d + 6c) of
//                        plane k = bit k of count(source d, colour c); d = 0 is the centre,
//                        d = 1..5 the factory displays.  Bit index == action index mod 30
//                        (game_runner.py:102-103), so "source holds colour" for the legal mask
//                        is PL0|PL1|PL2 and a display empties with three ANDs.
//   3     MISC           [4:0] plane 3 of the centre counts (centre can hold 15 of a colour)
//                        [5] first-player token in the centre (azul.py:71)
//                        [8:6] current_player  [11:9] next_first_player  (1-based, azul.py:27,37-43)
//                        [12] end_of_game  [15:13] sticky status (stuck, bag-empty, bad-import)
//                        [27:16] turn_counter (azul.py:30)
//   4     BOX            5 x 6-bit colour counts (azul.py:51; Lid pool only)
//   5     LID            5 x 6-bit colour counts (azul.py:52)
//   6     STEPS          env steps executed by this slot == position in the RNG schedule
//   per player p (5 words at 7 + 5p)
//   +0    PAT            pattern lines: row r at [6r+5:6r] = colour[2:0] | count[5:3]
//                        (one colour per row is an invariant of legal play, azul.py:171-173)
//   +1    WALL           bit (5*row + colour), the reference's colour-indexed wall (azul.py:23-24)
//   +2    SCF            [15:0] score (azul.py:26)  [18:16] floor count 0..7 (azul.py:25)
//   +3    STA            [11:0] first_player_stats  [27:12] -floor_penalty  [31:28] max_combo
//   +4    STB            [7:0] completed rows  [15:8] completed colours  [23:16] completed columns
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define AZB_HD __host__ __device__ __forceinline__
#define AZB_M __host__ __device__ __forceinline__
#define AZB_ROLLED _Pragma("unroll 1")   // keep rare, long paths small: the rollout kernel must fit the I-cache
#else
#define AZB_ROLLED
#define AZB_HD static inline
#define AZB_M inline
#endif

namespace azb {

enum : int { POOL_RANDOM = 0, POOL_LID = 1 };
enum : uint32_t { ST_ILLEGAL = 1, ST_ENDED = 2, ST_STUCK = 4, ST_BAG_EMPTY = 8, ST_BAD_IMPORT = 16 };
enum : uint32_t { PURPOSE_ACTION = 0, PURPOSE_REFILL = 1, PURPOSE_FIRST = 2, PURPOSE_RESET_REFILL = 3 };

// ---- intrinsics that exist on both sides ---------------------------------------------------
AZB_HD uint32_t mulhi(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
AZB_HD int popc(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
// count trailing zeros, 32 for x == 0
AZB_HD int ctz(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __clz((int)__brev(x));
#else
    return x ? __builtin_ctz(x) : 32;
#endif
}
// count leading zeros, 32 for x == 0
AZB_HD int clz(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __clz((int)x);
#else
    return x ? __builtin_clz(x) : 32;
#endif
}

constexpr uint32_t M6 = 0x01041041u;     // bits 0,6,12,18,24: the five colour slots of one source
constexpr uint32_t M5 = 0x00108421u;     // bits 0,5,10,15,20: one column of a 5x5 bit matrix
constexpr uint32_t PLANE_MASK = 0x3FFFFFFFu;

// 5 contiguous bits -> stride 6 (bit c -> bit 6c); the 25 partial products never collide
AZB_HD uint32_t spread5to6(uint32_t x) { return (x * M5) & M6; }
// stride 6 -> 5 contiguous bits (bit 6c -> bit c)
AZB_HD uint32_t gather6to5(uint32_t x) { return (((x & M6) * M5) >> 20) & 31u; }

// ---- Philox4x32-10 (Salmon et al. SC'11), the counter-based generator of the draw schedule ----
struct Philox {
    uint32_t k0, k1;
    AZB_M void operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) const
    {
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; r++) {
            uint32_t hi0 = mulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            uint32_t hi1 = mulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            c0 = hi1 ^ c1 ^ a; c1 = lo1; c2 = hi0 ^ c3 ^ b; c3 = lo0;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    }
};

// ---- the game in registers ----------------------------------------------------------------
template <int P>
struct Game {
    // In registers the fourth plane of the centre counts is held spread like the other planes (pl3: bit 6c = bit 3 of the
    // centre's count of colour c) and MISC[4:0] is zero; load / store convert from / to the packed word.
    uint32_t pl0, pl1, pl2, pl3, misc, box, lid, steps;
    uint32_t pat[P], wall[P], scf[P], sta[P], stb[P];

    static constexpr int WORDS = 7 + 5 * P;
    static constexpr int PLAYERS = P;

    AZB_M void load(const uint32_t* __restrict__ s, int64_t stride, int64_t g)
    {
        pl0 = s[0 * stride + g]; pl1 = s[1 * stride + g]; pl2 = s[2 * stride + g];
        set_misc_word(s[3 * stride + g]); box = s[4 * stride + g]; lid = s[5 * stride + g];
        steps = s[6 * stride + g];
#pragma unroll
        for (int p = 0; p < P; p++) {
            pat[p] = s[(7 + 5 * p) * stride + g];  wall[p] = s[(8 + 5 * p) * stride + g];
            scf[p] = s[(9 + 5 * p) * stride + g];  sta[p] = s[(10 + 5 * p) * stride + g];
            stb[p] = s[(11 + 5 * p) * stride + g];
        }
    }
    AZB_M void store(uint32_t* __restrict__ s, int64_t stride, int64_t g) const
    {
        s[0 * stride + g] = pl0; s[1 * stride + g] = pl1; s[2 * stride + g] = pl2;
        s[3 * stride + g] = misc_word(); s[4 * stride + g] = box; s[5 * stride + g] = lid;
        s[6 * stride + g] = steps;
#pragma unroll
        for (int p = 0; p < P; p++) {
            s[(7 + 5 * p) * stride + g] = pat[p];  s[(8 + 5 * p) * stride + g] = wall[p];
            s[(9 + 5 * p) * stride + g] = scf[p];  s[(10 + 5 * p) * stride + g] = sta[p];
            s[(11 + 5 * p) * stride + g] = stb[p];
        }
    }

    // the packed MISC word <-> misc + pl3
    AZB_M void set_misc_word(uint32_t w) { misc = w & ~31u; pl3 = ((w & 31u) * 0x00108421u) & 0x01041041u; }
    AZB_M uint32_t misc_word() const { return misc | ((((pl3 & 0x01041041u) * 0x00108421u) >> 20) & 31u); }
    AZB_M uint32_t sources() const { return pl0 | pl1 | pl2 | pl3; }    // bit d + 6c: source d holds colour c

    AZB_M uint32_t current_player() const { return (misc >> 6) & 7u; }
    AZB_M uint32_t next_first_player() const { return (misc >> 9) & 7u; }
    AZB_M bool ended() const { return (misc >> 12) & 1u; }
    AZB_M uint32_t status() const { return ((misc >> 13) & 7u) << 2; }
    AZB_M uint32_t turn_counter() const { return (misc >> 16) & 0xFFFu; }
    AZB_M void set_current_player(uint32_t v) { misc = (misc & ~(7u << 6)) | (v << 6); }
    AZB_M void set_next_first_player(uint32_t v) { misc = (misc & ~(7u << 9)) | (v << 9); }
    AZB_M void add_status(uint32_t bits) { misc |= ((bits >> 2) & 7u) << 13; }
    // python indexing with current_player-1: seat 0 wraps to the last player (azul.py:27)
    AZB_M int seat() const { uint32_t c = current_player(); return c ? (int)c - 1 : P - 1; }

    AZB_M uint32_t sel(const uint32_t (&a)[P], int s) const
    {
        uint32_t v = a[0];
#pragma unroll
        for (int p = 1; p < P; p++) v = (s == p) ? a[p] : v;
        return v;
    }
    AZB_M void put(uint32_t (&a)[P], int s, uint32_t v)
    {
#pragma unroll
        for (int p = 0; p < P; p++) a[p] = (s == p) ? v : a[p];
    }
};

// ---- legal mask: check_all_valid (game_runner.py:113-117) over is_legal_move (azul.py:162-176) ----
// legal(d,c,p) = source d holds colour c  AND  (p == 0 OR (row p-1 of the mover holds no other
// colour AND wall[p-1][c] is clear)).  A row already full of c stays legal (azul.py:171-175).
template <int P>
AZB_HD void legal_mask(const Game<P>& g, uint32_t m[6])
{
    const uint32_t src = g.sources();
    const int s = g.seat();
    const uint32_t pat = g.sel(g.pat, s), wall = g.sel(g.wall, s);
    m[0] = src;
#pragma unroll
    for (int r = 0; r < 5; r++) {
        const uint32_t cnt = (pat >> (6 * r + 3)) & 7u, col = (pat >> (6 * r)) & 7u;
        const uint32_t allowed = (cnt ? (1u << col) : 31u) & ~(wall >> (5 * r)) & 31u;
        m[r + 1] = src & (spread5to6(allowed) * 63u);
    }
}

// The destination half of the legal mask as one word per player: bit 6c + r = colour c may still go to pattern line r
// (the line is empty or holds c, and wall[r][c] is clear; azul.py:171-175), so that (open >> r) & M6 is line r's colour
// set already spread to the source planes' stride.  The rollout keeps these words in registers: a move into line r
// leaves exactly {c} open there, scoring rebuilds them (rollout_steps).
template <int P>
AZB_HD uint32_t open_rows(const Game<P>& g, int pl)
{
    const uint32_t pat = g.pat[pl], wall = g.wall[pl];
    uint32_t o = 0;
#pragma unroll
    for (int r = 0; r < 5; r++) {
        const uint32_t cnt = (pat >> (6 * r + 3)) & 7u, col = (pat >> (6 * r)) & 7u;
        o |= spread5to6((cnt ? (1u << col) : 31u) & ~(wall >> (5 * r)) & 31u) << r;
    }
    return o;
}
// legal_mask from the open-rows words (same result as legal_mask(g, m) when open[p] == open_rows(g, p))
template <int P>
AZB_HD void legal_mask_open(const Game<P>& g, const uint32_t (&open)[P], uint32_t m[6])
{
    const uint32_t src = g.sources();
    const uint32_t o = g.sel(open, g.seat());
    m[0] = src;
    m[1] = src & ((o & M6) * 63u);
    m[2] = src & (((o >> 1) & M6) * 63u);
    m[3] = src & (((o >> 2) & M6) * 63u);
    m[4] = src & (((o >> 3) & M6) * 63u);
    m[5] = src & (((o >> 4) & M6) * 63u);
}

// floors[] += n capped at 7 (azul.py:119-123)
AZB_HD uint32_t floor_add(uint32_t scf, uint32_t n)
{
    uint32_t f = ((scf >> 16) & 7u) + n;
    f = f < 7u ? f : 7u;
    return (scf & ~(7u << 16)) | (f << 16);
}

// ---- move (azul.py:118-161); no legality check, like the reference ----
// p = destination (0 floor, 1..5 pattern line), b = d + 6c = the bit of (source d, colour c) in the planes.
// Branch-free: a warp holds 32 different games, so "display or centre" and "pattern line or floor" are selects, not
// branches.  A centre take is the display case with an empty "rest".
template <int P, int POOL, bool TRACK>
AZB_HD void apply_move_core(Game<P>& g, uint32_t p, uint32_t b, uint32_t* open)
{
    const uint32_t c = (b * 43u) >> 8, c6 = 6u * c, d = b - c6;       // b < 30: b / 6 == (b * 43) >> 8
    const int s = g.seat();
    const bool centre = d == 0u;
    const uint32_t cbit = 1u << c6;
    // the planes moved down by d: bit 6c' = (source d, colour c'); pl3 only has bits at d = 0
    const uint32_t t0 = g.pl0 >> d, t1 = g.pl1 >> d, t2 = g.pl2 >> d, t3 = g.pl3 >> d;
    // tiles taken, still in place: n * cbit
    const uint32_t n6 = (t3 & cbit) * 8u + ((t2 & cbit) * 4u + ((t1 & cbit) * 2u + (t0 & cbit)));
    const uint32_t n = n6 >> c6;
    // azul.py:125-133: the chosen colour leaves, the rest of display d joins the centre -- a bit-sliced
    // 4-bit ripple add over all five colours at once.  azul.py:134-138: from the centre only colour c leaves.
    const uint32_t others = M6 & ~cbit;
    const uint32_t rest = centre ? 0u : others, keepc = centre ? others : M6;
    const uint32_t r0 = t0 & rest, r1 = t1 & rest, r2 = t2 & rest;
    const uint32_t k0 = g.pl0 & r0;
    const uint32_t k1 = (g.pl1 & r1) | (k0 & (g.pl1 ^ r1));
    const uint32_t k2 = (g.pl2 & r2) | (k1 & (g.pl2 ^ r2));
    const uint32_t clear = ~((M6 << d) | M6);            // the emptied display (or nothing more, d = 0) and the old centre
    g.pl0 = (g.pl0 & clear) | ((g.pl0 ^ r0) & keepc);
    g.pl1 = (g.pl1 & clear) | ((g.pl1 ^ r1 ^ k0) & keepc);
    g.pl2 = (g.pl2 & clear) | ((g.pl2 ^ r2 ^ k1) & keepc);
    g.pl3 = (g.pl3 ^ k2) & keepc;
    // azul.py:139-143: the first-player token goes with the first centre take, onto the floor first;
    // next_first_player [11:9] := current_player [8:6]
    const uint32_t t32 = centre ? (g.misc & 32u) : 0u;
    const uint32_t nf_mask = t32 * 112u;                  // 0xE00 when the token moves
    const uint32_t misc = g.misc ^ t32;
    g.misc = (misc & ~nf_mask) | ((misc << 3) & nf_mask);
    // azul.py:145-161: fill row p-1 up to its capacity p, the rest (everything when p = 0) falls to the floor
    const bool to_row = p != 0u;
    const uint32_t pat = g.sel(g.pat, s);
    const uint32_t r = to_row ? p - 1u : 0u, sh = 6u * r;
    const uint32_t cnt = (pat >> (sh + 3u)) & 7u;
    const uint32_t room = p - cnt;                       // >= 0 when to_row
    const uint32_t placed = to_row ? (n < room ? n : room) : 0u;
    const uint32_t to_floor = n - placed;
    const uint32_t pw = 1u << sh;
    // to_row: cnt + placed >= 1 (a tile was placed, or the line was already full), so the colour is always written
    const uint32_t field = (cnt + placed) * 8u + c;
    const uint32_t newpat = (pat & ~(pw * 63u)) | field * pw;
    g.put(g.pat, s, to_row ? newpat : pat);
    // floors[] += n capped at 7 (azul.py:119-123): both candidates share the score bits, so min() compares the floor fields
    const uint32_t scf = g.sel(g.scf, s);
    const uint32_t added = t32 * 2048u + (to_floor * 65536u + scf), capped = scf | (7u << 16);
    g.put(g.scf, s, added < capped ? added : capped);
    if (POOL == POOL_LID) g.lid += to_floor * cbit;                  // azul.py:156-157,160-161
    if (TRACK) {                                                      // open rows of the mover: line p-1 now takes only c
        const uint32_t pr = 1u << r;
        const uint32_t line = pr * M6, only = pr * cbit;
#pragma unroll
        for (int q = 0; q < P; q++) {
            const uint32_t o = open[q];
            open[q] = (to_row && s == q) ? ((o & ~line) | only) : o;
        }
    }
}
template <int P, int POOL>
AZB_HD void apply_move(Game<P>& g, uint32_t action)
{
    const uint32_t p = action / 30u;
    apply_move_core<P, POOL, false>(g, p, action - 30u * p, nullptr);
}

// azul.py:177-181 (GT: Game<P>, or the factory-count variant's GameV<P,F>, which shares the per-player words)
template <class GT>
AZB_HD void next_player(GT& g)
{
    const uint32_t c = g.current_player();
    g.set_current_player(c < (uint32_t)GT::PLAYERS ? c + 1u : 1u);
}

// azul.py:182-183 -- every display and all six centre slots (token included) are empty
template <int P>
AZB_HD bool is_end_of_round(const Game<P>& g)
{
    return (g.sources() | (g.misc & 32u)) == 0u;
}

// azul.py:184-191 -- some wall row of some player holds all five colours
template <class GT>
AZB_HD bool is_end_of_game(const GT& g)
{
    uint32_t any = 0;
#pragma unroll
    for (int p = 0; p < GT::PLAYERS; p++) {
        const uint32_t w = g.wall[p];
        uint32_t t = w & (w >> 1);
        t &= t >> 2;
        t &= w >> 4;
        any |= t & M5;
    }
    return any != 0u;
}

// ---- count_score (azul.py:192-295) for one player ----
// Adjacency runs on a column-space copy of the wall (column = (colour + row) mod 5,
// azul.py:194-196) with ctz/clz run-length counts instead of the reference's four walks.
template <int POOL, class GT>
AZB_HD void score_player_g(GT& g, const int pl)
{
    uint32_t scf = g.scf[pl], pat = g.pat[pl], wall = g.wall[pl], sta = g.sta[pl], stb = g.stb[pl];
    // count_floor, azul.py:200-210: 0,-1,-2,-4,-6,-8,-11,-14
    const uint32_t f = (scf >> 16) & 7u;
    const uint32_t pen = (0xEB864210u >> (4u * f)) & 15u;
    int32_t gain = -(int32_t)pen;
    sta += pen << 12;                                             // floor_penalty statistic (:208)
    uint32_t wc = 0;                                              // wall in column space
#pragma unroll
    for (int r = 0; r < 5; r++) {
        const uint32_t row = (wall >> (5 * r)) & 31u;
        wc |= (((row << r) | (row >> (5 - r))) & 31u) << (5 * r);
    }
    uint32_t combo = sta >> 28;
    // the full lines (:216, count == row + 1), ascending: a warp walks max-over-lanes(#full lines) iterations instead
    // of all five rows (nearly every row is full in SOME of a warp's 32 games)
    uint32_t full = 0;
#pragma unroll
    for (int r = 0; r < 5; r++) full |= (((pat >> (6 * r + 3)) & 7u) == (uint32_t)(r + 1) ? 1u : 0u) << r;
    AZB_ROLLED
    while (full) {
        const uint32_t r = (uint32_t)ctz(full);
        full &= full - 1u;
        const uint32_t sh6 = 6u * r, sh5 = 5u * r;
        const uint32_t c = (pat >> sh6) & 7u;
        {
            pat &= ~(63u << sh6);                                 // :218
            wall |= 1u << (sh5 + c);                              // :219
            if (POOL == POOL_LID) g.lid += r << (6u * c);         // :220-222
            uint32_t k = c + r;
            k = k >= 5u ? k - 5u : k;                             // to_wall_position, :194-196
            wc |= 1u << (sh5 + k);
            const uint32_t rowbits = (wc >> sh5) & 31u;
            const int hr = ctz(~(rowbits >> (k + 1u)));           // :230-236 walk right
            const int hl = clz(~((rowbits << (31u - k)) << 1));   // :237-242 walk left
            const uint32_t colbits = (wc >> k) & M5;              // column k, bit 5j = row j
            const int vd = (ctz(~(colbits >> (sh5 + 5u)) & M5) * 13) >> 6;                 // :244-250 walk down
            const int vu = (clz(~((colbits << (31u - sh5)) << 5) & 0x84210800u) * 13) >> 6;  // :251-257 walk up
            const int h = hr + hl, v = vd + vu;
            const int pts = h + v + 1 + ((h > 0 && v > 0) ? 1 : 0);   // :258-263
            combo = (uint32_t)pts > combo ? (uint32_t)pts : combo;    // :264
            gain += pts;
            if (rowbits == 31u) { gain += 2; stb += 1u; }                       // :266-272
            if (((wall >> c) & M5) == M5) { gain += 10; stb += 1u << 8; }       // :274-280
            if (colbits == M5) { gain += 7; stb += 1u << 16; }                  // :282-288
        }
    }
    int32_t score = (int32_t)(scf & 0xFFFFu) + gain;              // :292
    score = score < 0 ? 0 : score;                                // :294-295
    g.scf[pl] = (uint32_t)score;                                  // floor cleared (:209)
    g.pat[pl] = pat; g.wall[pl] = wall;
    g.sta[pl] = (sta & 0x0FFFFFFFu) | (combo << 28);
    g.stb[pl] = stb;
}

template <int P, int POOL>
AZB_HD void score_player(Game<P>& g, const int pl) { score_player_g<POOL>(g, pl); }

template <int POOL, class GT>
AZB_HD void count_score_g(GT& g)
{
#pragma unroll
    for (int p = 0; p < GT::PLAYERS; p++) score_player_g<POOL>(g, p);
}
template <int P, int POOL>
AZB_HD void count_score(Game<P>& g) { count_score_g<POOL>(g); }

// one more tile of colour c on source position b = d + 6c: bit-sliced increment
AZB_HD void plane_inc(uint32_t& pl0, uint32_t& pl1, uint32_t& pl2, uint32_t b)
{
    const uint32_t t = 1u << b;
    const uint32_t k0 = pl0 & t; pl0 ^= t;
    const uint32_t k1 = pl1 & k0; pl1 ^= k0;
    pl2 ^= k1;
}

// azul.py:64-73: everything new_round does before the 20 draws
template <int P>
AZB_HD void new_round_header(Game<P>& g)
{
    const uint32_t nf = g.next_first_player();
    g.set_current_player(nf);                                     // :66
    const int s = nf ? (int)nf - 1 : P - 1;
#pragma unroll
    for (int p = 0; p < P; p++) g.sta[p] += (s == p) ? 1u : 0u;   // :67 first_player_stats
    g.misc = (g.misc & ~(0xFFFu << 16)) | (((g.turn_counter() + 1u) & 0xFFFu) << 16);   // :68
    g.set_next_first_player(0u);                                  // :69
    g.misc |= 32u;                                                // :71 centre empty + token
    g.pl0 = g.pl1 = g.pl2 = g.pl3 = 0u;                           // :73
}

// Lid pool: the box for the duration of a refill, held as the four cumulative counts the draw compares against
// (e0 = box[0], e1 = box[0] + box[1], ...) packed as the four bytes of ONE register, each with its bit 7 set, and the
// total.  A draw compares its point with all four thresholds in one subtraction (byte j of E - (r + 1) * 0x01010101
// keeps bit 7 exactly when e_j > r; no byte borrows because 128 + e_j - r - 1 stays in [0, 255]) and lowers the
// thresholds above the point in one more.  A real game holds 100 tiles, so a cumulative count fits 7 bits; a
// box with more than 127 tiles (only reachable from an imported record that no game can produce) is flagged
// ST_BAD_IMPORT by the caller and clamped.
struct BoxRegs {
    uint32_t E, total;
    // returns false when the counts do not fit (more than 127 tiles)
    AZB_M bool unpack(uint32_t w)
    {
        const uint32_t e0 = w & 63u, e1 = e0 + ((w >> 6) & 63u), e2 = e1 + ((w >> 12) & 63u), e3 = e2 + ((w >> 18) & 63u);
        total = e3 + ((w >> 24) & 63u);
        const bool fits = total <= 127u;
        const uint32_t c0 = e0 < 127u ? e0 : 127u, c1 = e1 < 127u ? e1 : 127u, c2 = e2 < 127u ? e2 : 127u, c3 = e3 < 127u ? e3 : 127u;
        total = fits ? total : 127u;
        E = c0 | (c1 << 8) | (c2 << 16) | (c3 << 24) | 0x80808080u;
        return fits;
    }
    AZB_M uint32_t pack() const
    {
        const uint32_t e0 = E & 127u, e1 = (E >> 8) & 127u, e2 = (E >> 16) & 127u, e3 = (E >> 24) & 127u;
        return e0 | ((e1 - e0) << 6) | ((e2 - e1) << 12) | ((e3 - e2) << 18) | ((total - e3) << 24);
    }
};

// one draw from a non-empty box (azul.py:87-89): colour c <=> e(c-1) <= r < e(c) for the point r = mulhi(x, total);
// taking one tile of c lowers every threshold from e(c) on.  Returns the colour.
AZB_HD uint32_t lid_draw_fast(BoxRegs& B, uint32_t& x)
{
    const uint64_t prod = (uint64_t)x * B.total;                  // one wide multiply: the point and the next x
    const uint32_t r = (uint32_t)(prod >> 32);
    x = (uint32_t)prod;
    const uint32_t above = ((B.E - (r + 1u) * 0x01010101u) >> 7) & 0x01010101u;    // byte j = 1 when e_j > r
    B.E -= above;
    B.total -= 1u;
    return 4u - ((above * 0x01010101u) >> 24);
}

// Lid pool, one draw (azul.py:79-89): pour the lid into an empty box first.  Returns colour or -1 when no tile is left.
template <class GT>
AZB_HD int lid_draw(GT& g, BoxRegs& B, uint32_t& x)
{
    if (B.total == 0u) {                                          // :81-83
        if (!B.unpack(g.lid)) g.add_status(ST_BAD_IMPORT);
        g.lid = 0u;
        if (B.total == 0u) { g.add_status(ST_BAG_EMPTY); return -1; }   // :86 TODO in the reference
    }
    return (int)lid_draw_fast(B, x);
}

// azul.py:64-89 with the Philox draw schedule (DESIGN.md "RNG schedule"): call j of
// Philox(gid, steps, purpose, j) yields words R[4j..4j+3]; Random pool: display i draws its four
// colours from R[i] (c = mulhi(x,5), x *= 5); Lid pool: display i draws two colours from each of
// R[2i], R[2i+1] (r = mulhi(x,total), x *= total).
template <int P, int POOL>
AZB_HD void new_round_philox(Game<P>& g, const Philox& rng, uint32_t gid, uint32_t purpose)
{
    new_round_header(g);
    constexpr uint32_t CALLS = POOL == POOL_LID ? 3u : 2u;
    BoxRegs B;
    if (POOL == POOL_LID) { if (!B.unpack(g.box)) g.add_status(ST_BAD_IMPORT); }
    AZB_ROLLED
    for (uint32_t j = 0; j < CALLS; j++) {
        uint32_t w[4];
        rng(gid, g.steps, purpose, j, w);
        if (POOL == POOL_RANDOM) {
            const uint32_t nq = j == 0u ? 4u : 1u;                // displays 0..3 from call 0, display 4 from call 1
            AZB_ROLLED
            for (uint32_t q = 0; q < nq; q++) {
                uint32_t x = q == 0u ? w[0] : q == 1u ? w[1] : q == 2u ? w[2] : w[3];
                const uint32_t d = 4u * j + q + 1u;
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    const uint32_t c = mulhi(x, 5u);              // :78 randrange(0,5)
                    x *= 5u;
                    plane_inc(g.pl0, g.pl1, g.pl2, d + 6u * c);
                }
            }
        } else {
            const uint32_t nh = j == 2u ? 2u : 4u;                // half-displays: words 2i, 2i+1 of display i
#pragma unroll
            for (uint32_t q = 0; q < 4u; q++) {
                if (q < nh) {
                    uint32_t x = w[q];
                    const uint32_t d = 2u * j + (q >> 1) + 1u;
                    if (B.total >= 2u) {                          // no refill inside this pair: two unchecked draws
                        const uint32_t c0 = lid_draw_fast(B, x), c1 = lid_draw_fast(B, x);
                        plane_inc(g.pl0, g.pl1, g.pl2, d + 6u * c0);
                        plane_inc(g.pl0, g.pl1, g.pl2, d + 6u * c1);
                    } else {
                        AZB_ROLLED
                        for (int t = 0; t < 2; t++) {
                            const int c = lid_draw(g, B, x);
                            if (c >= 0) plane_inc(g.pl0, g.pl1, g.pl2, d + 6u * (uint32_t)c);
                        }
                    }
                }
            }
        }
    }
    if (POOL == POOL_LID) g.box = B.pack();
}

// azul.py:64-89 with the 20 colours injected (replay of recorded draws; -1 leaves a slot empty)
template <int P, int POOL, typename DrawFn>
AZB_HD void new_round_injected(Game<P>& g, DrawFn draw)
{
    new_round_header(g);
#pragma unroll 1
    for (int k = 0; k < 20; k++) {
        const int c = draw(k);
        if (c < 0 || c > 4) continue;
        if (POOL == POOL_LID) {
            const uint32_t tot = (g.box & 63u) + ((g.box >> 6) & 63u) + ((g.box >> 12) & 63u) +
                                 ((g.box >> 18) & 63u) + ((g.box >> 24) & 63u);
            if (tot == 0u) { g.box = g.lid; g.lid = 0u; }         // :81-83
            if (((g.box >> (6 * c)) & 63u) == 0u) { g.add_status(ST_BAG_EMPTY); continue; }
            g.box -= 1u << (6 * c);                               // :89
        }
        plane_inc(g.pl0, g.pl1, g.pl2, (uint32_t)(k / 4 + 1) + 6u * (uint32_t)c);
    }
}

// Azul.__init__ (azul.py:18-61): an empty game that still needs new_round()
template <int P, int POOL>
AZB_HD void init_game(Game<P>& g, uint32_t first_player)
{
    g.pl0 = g.pl1 = g.pl2 = g.pl3 = 0u;
    g.misc = first_player << 9;
    g.box = (POOL == POOL_LID) ? (20u | 20u << 6 | 20u << 12 | 20u << 18 | 20u << 24) : 0u;
    g.lid = 0u;
#pragma unroll
    for (int p = 0; p < P; p++) { g.pat[p] = g.wall[p] = g.scf[p] = g.sta[p] = g.stb[p] = 0u; }
}

// fresh game in this slot: Azul(rules) + new_round() (game_runner.py:79-80)
template <int P, int POOL>
AZB_HD void reset_game(Game<P>& g, const Philox& rng, uint32_t gid, int first_rule)
{
    uint32_t first = (uint32_t)first_rule;
    if (first_rule == 0) {                                        // azul.py:36-37 random.choice
        uint32_t w[4];
        rng(gid, g.steps, PURPOSE_FIRST, 0u, w);
        first = 1u + mulhi(w[0], (uint32_t)P);
    }
    init_game<P, POOL>(g, first);
    new_round_philox<P, POOL>(g, rng, gid, PURPOSE_RESET_REFILL);
}

// ---- step (azul.py:296-313) after the legality / ended checks; returns true when the game ended ----
template <int P, int POOL, typename RefillFn>
AZB_HD bool advance(Game<P>& g, uint32_t action, RefillFn refill)
{
    apply_move<P, POOL>(g, action);                               // :304
    g.steps += 1u;
    if (is_end_of_round(g)) {                                     // :306
        count_score<P, POOL>(g);                                  // :307
        if (is_end_of_game(g)) { g.misc |= 1u << 12; return true; }   // :308-309
        refill(g);                                                // :311
    } else {
        next_player(g);                                           // :313
    }
    return false;
}

AZB_HD bool action_is_legal(const uint32_t m[6], uint32_t action)
{
    if (action >= 180u) return false;
    const uint32_t p = action / 30u, b = action - 30u * p;
    uint32_t w = m[0];
#pragma unroll
    for (int i = 1; i < 6; i++) w = (p == (uint32_t)i) ? m[i] : w;
    return (w >> b) & 1u;
}

// is_legal_move (azul.py:162-176) for one action, without building the 180-bit mask; same result as
// action_is_legal(legal_mask(g), action)
template <int P>
AZB_HD bool move_is_legal(const Game<P>& g, uint32_t action)
{
    // branch-free: a warp tests 32 different games
    const uint32_t a = action < 180u ? action : 0u;
    const uint32_t p = a / 30u, b = a - 30u * p, c = b / 6u;
    const uint32_t src = g.sources();
    const int s = g.seat();
    const uint32_t pat = g.sel(g.pat, s), wall = g.sel(g.wall, s);
    const uint32_t r = p ? p - 1u : 0u, cnt = (pat >> (6u * r + 3u)) & 7u, col = (pat >> (6u * r)) & 7u;
    const bool source_ok = (src >> b) & 1u;                                           // azul.py:164-169
    const bool row_ok = ((cnt == 0u) | (col == c)) & !((wall >> (5u * r + c)) & 1u);   // azul.py:171-175
    return (action < 180u) & source_ok & ((p == 0u) | row_ok);                        // the floor takes anything
}

// is_legal_move + move for one supplied action (Azul.step, azul.py:301-304): returns false and leaves the game untouched
// when the action is illegal.  One decode of the action and one pick of the mover's words serve both halves.
template <int P, int POOL>
AZB_HD bool move_if_legal(Game<P>& g, uint32_t action)
{
    const uint32_t a = action < 180u ? action : 0u;
    const uint32_t p = a / 30u, b = a - 30u * p, c = (b * 43u) >> 8;
    const int s = g.seat();
    const uint32_t pat = g.sel(g.pat, s), wall = g.sel(g.wall, s);
    const uint32_t r = p ? p - 1u : 0u, cnt = (pat >> (6u * r + 3u)) & 7u, col = (pat >> (6u * r)) & 7u;
    const bool source_ok = (g.sources() >> b) & 1u;                                   // azul.py:164-169
    const bool row_ok = ((cnt == 0u) | (col == c)) & !((wall >> (5u * r + c)) & 1u);   // azul.py:171-175
    const bool legal = (action < 180u) & source_ok & ((p == 0u) | row_ok);            // the floor takes anything
    if (legal) apply_move_core<P, POOL, false>(g, p, b, nullptr);
    return legal;
}

// position of the k-th (0-based) set bit of a 30-bit word; k < popc(m).  Binary search: at each level, when k is at least
// the popcount c of the low half, the bit lies in the high half: skip the low half and look for the (k - c)-th bit there.
AZB_HD uint32_t select_bit(uint32_t m, uint32_t k)
{
    uint32_t pos = 0, c;
    c = (uint32_t)popc(m & 0xFFFFu); if (k >= c) { k -= c; pos += 16; m >>= 16; }
    c = (uint32_t)popc(m & 0xFFu);   if (k >= c) { k -= c; pos += 8;  m >>= 8; }
    c = (uint32_t)popc(m & 0xFu);    if (k >= c) { k -= c; pos += 4;  m >>= 4; }
    c = (uint32_t)popc(m & 0x3u);    if (k >= c) { k -= c; pos += 2;  m >>= 2; }
    c = m & 1u;                      if (k >= c) { pos += 1; }
    return pos;
}

// The integer random agent (game_runner.py:87-97): legal floor actions (p = 0) weigh 1, every
// other legal action 100; the point r = mulhi(word, total) walks words 1..5 first, then word 0.
// Yields the action as destination p and plane bit b (action = 30 p + b); false when no action is legal.
// Branch-free up to the final bit select.
AZB_HD bool random_action_pb(const uint32_t m[6], uint32_t word, uint32_t& p, uint32_t& b)
{
    const uint32_t n1 = (uint32_t)popc(m[1]), n2 = (uint32_t)popc(m[2]), n3 = (uint32_t)popc(m[3]),
                   n4 = (uint32_t)popc(m[4]), n5 = (uint32_t)popc(m[5]), n0 = (uint32_t)popc(m[0]);
    const uint32_t e1 = n1, e2 = e1 + n2, e3 = e2 + n3, e4 = e3 + n4, n_hi = e4 + n5;
    const uint32_t total = 100u * n_hi + n0;
    const uint32_t r = mulhi(word, total);
    const bool heavy = r < 100u * n_hi;
    const uint32_t kh = r / 100u;                        // rank among the heavy actions
    // word i + 1 holds the kh-th heavy action: the thresholds are monotone, so four predicated overwrites pick the
    // word, its destination and the rank before it (an `i == k ? ... :` chain compiles to a divergent switch)
    const bool g1 = kh >= e1, g2 = kh >= e2, g3 = kh >= e3, g4 = kh >= e4;
    uint32_t before = 0u, wh = m[1], ph = 1u;
    before = g1 ? e1 : before; wh = g1 ? m[2] : wh; ph = g1 ? 2u : ph;
    before = g2 ? e2 : before; wh = g2 ? m[3] : wh; ph = g2 ? 3u : ph;
    before = g3 ? e3 : before; wh = g3 ? m[4] : wh; ph = g3 ? 4u : ph;
    before = g4 ? e4 : before; wh = g4 ? m[5] : wh; ph = g4 ? 5u : ph;
    const uint32_t w = heavy ? wh : m[0];
    const uint32_t k = heavy ? kh - before : r - 100u * n_hi;
    p = heavy ? ph : 0u;
    b = select_bit(w, k);
    return total != 0u;
}
// the same as an action index; 180 when no action is legal
AZB_HD uint32_t random_action(const uint32_t m[6], uint32_t word)
{
    uint32_t p, b;
    return random_action_pb(m, word, p, b) ? 30u * p + b : 180u;
}

// The wall points (azul.py:211-290, without the bonus statistics) that the full pattern lines `full` (bit r = row r; its
// colour at (pat >> 6r) & 7) earn when placed in row order on the colour-indexed wall `wall` / its column-space copy `wc`.
// The placement arithmetic of score_player_g, kept separate so that the scoring pass's code stays as it is.
AZB_HD int wall_gain(uint32_t pat, uint32_t wall, uint32_t wc, uint32_t full)
{
    int gain = 0;
    AZB_ROLLED
    while (full) {
        const uint32_t r = (uint32_t)ctz(full);
        full &= full - 1u;
        const uint32_t sh5 = 5u * r, c = (pat >> (6u * r)) & 7u;
        wall |= 1u << (sh5 + c);
        uint32_t k = c + r;
        k = k >= 5u ? k - 5u : k;
        wc |= 1u << (sh5 + k);
        const uint32_t rowbits = (wc >> sh5) & 31u;
        const int hr = ctz(~(rowbits >> (k + 1u)));
        const int hl = clz(~((rowbits << (31u - k)) << 1));
        const uint32_t colbits = (wc >> k) & M5;
        const int vd = (ctz(~(colbits >> (sh5 + 5u)) & M5) * 13) >> 6;
        const int vu = (clz(~((colbits << (31u - sh5)) << 5) & 0x84210800u) * 13) >> 6;
        const int h = hr + hl, v = vd + vu;
        gain += h + v + 1 + ((h > 0 && v > 0) ? 1 : 0);
        gain += rowbits == 31u ? 2 : 0;
        gain += ((wall >> c) & M5) == M5 ? 10 : 0;
        gain += colbits == M5 ? 7 : 0;
    }
    return gain;
}

// ---- the greedy agent: the best one-move score for the seat to move ----
// Spec (shared with ao_greedy_action in tests/harness/greedy_oracle.c):
//   v(a) = the mover's score after Azul.move(a) (azul.py:118-161) and count_score (azul.py:192-295) on a copy, WITHOUT the
//          clamp at zero of azul.py:294-295: score + the wall points and bonuses of every full pattern line placed in row
//          order - the floor penalty.  (With the clamp, at score 0 dumping tiles to the floor would tie with a placement.)
//   T    = the legal actions of largest v, in ascending action index.
//   pick = T[mulhi(word, |T|)], word = the random agent's word of this env step (word steps & 3 of
//          Philox(gid, steps >> 2, ACTION, 0)); one best action uses no randomness.  180 when no action is legal.
// v differs between actions only through the floor after the move and, for a move that completes line r with colour c,
// the wall points with (r, c) added: so the value compared is u = (completes ? W(r, c) - W0 : 0) - penalty(floor after),
// with W0 the wall points of the lines already full and W(r, c) computed once per (line, colour) that some source can
// complete.  One game per thread: the loops run over colours and the sources holding them, never over all 180 actions.
template <int P, int POOL>
AZB_HD uint32_t greedy_action(const Game<P>& g, const uint32_t m[6], uint32_t word)
{
    const int s = g.seat();
    const uint32_t pat = g.sel(g.pat, s), wall = g.sel(g.wall, s), scf = g.sel(g.scf, s);
    const uint32_t f = (scf >> 16) & 7u, token = (g.misc >> 5) & 1u;
    uint32_t wc = 0, full = 0;
    int room[5];
#pragma unroll
    for (int r = 0; r < 5; r++) {
        const uint32_t row = (wall >> (5 * r)) & 31u;
        wc |= (((row << r) | (row >> (5 - r))) & 31u) << (5 * r);
        room[r] = r + 1 - (int)((pat >> (6 * r + 3)) & 7u);
        full |= (room[r] == 0 ? 1u : 0u) << r;
    }
    const int w0 = wall_gain(pat, wall, wc, full);
    const uint32_t src = m[0];                           // every source / colour that holds a tile
    int best = -1000;
    uint32_t bm[6] = {0u, 0u, 0u, 0u, 0u, 0u};          // the legal actions of value `best`, as mask words
    AZB_ROLLED
    for (uint32_t c = 0; c < 5u; c++) {
        uint32_t bits = (src >> (6u * c)) & 63u;
        if (!bits) continue;
        // the counts of colour c in its sources; the largest decides which lines a take of c can complete
        int maxn = 0;
        for (uint32_t t = bits; t; t &= t - 1u) {
            const uint32_t b = (uint32_t)ctz(t) + 6u * c;
            const int n = (int)(((g.pl0 >> b) & 1u) | (((g.pl1 >> b) & 1u) << 1) | (((g.pl2 >> b) & 1u) << 2) | (((g.pl3 >> b) & 1u) << 3));
            maxn = n > maxn ? n : maxn;
        }
        int dw[5];
#pragma unroll
        for (int r = 0; r < 5; r++) {
            dw[r] = 0;
            // line r open for c (m[r + 1] holds c at some source) and completable by the largest take
            const bool open = ((m[r + 1] >> (6u * c)) & 63u) != 0u;
            if (open && room[r] > 0 && maxn >= room[r])
                dw[r] = wall_gain((pat & ~(7u << (6 * r))) | (c << (6 * r)), wall, wc, full | (1u << r)) - w0;
        }
        AZB_ROLLED
        for (; bits; bits &= bits - 1u) {
            const uint32_t d = (uint32_t)ctz(bits), b = d + 6u * c;
            const int n = (int)(((g.pl0 >> b) & 1u) | (((g.pl1 >> b) & 1u) << 1) | (((g.pl2 >> b) & 1u) << 2) | (((g.pl3 >> b) & 1u) << 3));
            const int f0 = (int)f + (d == 0u ? (int)token : 0);
            // the floor (p = 0) takes all n tiles; line r = p - 1 takes up to room[r], the rest falls
            int lbest = -1000;
            uint32_t lset = 0u;
#pragma unroll
            for (int p = 0; p < 6; p++) {
                const int rm = p == 0 ? 0 : room[p - 1];
                const int placed = p == 0 ? 0 : (n < rm ? n : rm);
                int fl = f0 + n - placed;
                fl = fl < 7 ? fl : 7;
                const int pen = (int)((0xEB864210u >> (4 * fl)) & 15u);
                const int u = (p > 0 && rm > 0 && n >= rm ? dw[p - 1] : 0) - pen;
                const bool legal = (m[p] >> b) & 1u;
                const bool gt = legal && u > lbest, eq = legal && u == lbest;
                lset = gt ? 1u << p : (eq ? lset | (1u << p) : lset);
                lbest = gt ? u : lbest;
            }
            // (the floor always takes a tile the source holds: lset is never empty)
            const bool gt = lbest > best, take = lbest >= best;
#pragma unroll
            for (int p = 0; p < 6; p++) {
                const uint32_t keep = gt ? 0u : bm[p];
                bm[p] = take ? keep | (((lset >> p) & 1u) << b) : bm[p];
            }
            best = gt ? lbest : best;
        }
    }
    // T in ascending action index: word 0 (the floor, actions 0..29) first, then lines 1..5
    const uint32_t n0 = (uint32_t)popc(bm[0]), n1 = (uint32_t)popc(bm[1]), n2 = (uint32_t)popc(bm[2]),
                   n3 = (uint32_t)popc(bm[3]), n4 = (uint32_t)popc(bm[4]), n5 = (uint32_t)popc(bm[5]);
    const uint32_t e1 = n0, e2 = e1 + n1, e3 = e2 + n2, e4 = e3 + n3, e5 = e4 + n4, total = e5 + n5;
    if (total == 0u) return 180u;
    const uint32_t k = mulhi(word, total);
    uint32_t before = 0u, w = bm[0], p = 0u;
    before = k >= e1 ? e1 : before; w = k >= e1 ? bm[1] : w; p = k >= e1 ? 1u : p;
    before = k >= e2 ? e2 : before; w = k >= e2 ? bm[2] : w; p = k >= e2 ? 2u : p;
    before = k >= e3 ? e3 : before; w = k >= e3 ? bm[3] : w; p = k >= e3 ? 3u : p;
    before = k >= e4 ? e4 : before; w = k >= e4 ? bm[4] : w; p = k >= e4 ? 4u : p;
    before = k >= e5 ? e5 : before; w = k >= e5 ? bm[5] : w; p = k >= e5 ? 5u : p;
    return 30u * p + select_bit(w, k - before);
}

// the opponent's pick at one env step: the random agent's, or the greedy agent's, from the same action word
template <int P, int POOL, bool GREEDY>
AZB_HD uint32_t opponent_pick(const Game<P>& g, const uint32_t m[6], uint32_t word)
{
    return GREEDY ? greedy_action<P, POOL>(g, m, word) : random_action(m, word);
}

// ---- unpacked record <-> packed game (kernel K7; record layout in layout.py) -----------------
// Returns false (and flags ST_BAD_IMPORT) when the record cannot be represented: a pattern row
// holding two colours, or a count outside its field.
template <int P, typename Rd>
AZB_HD bool import_record(Game<P>& g, Rd rd)
{
    bool ok = true;
    g.pl0 = g.pl1 = g.pl2 = g.pl3 = 0u; g.misc = 0u; g.box = g.lid = 0u;
    for (int i = 0; i < 5; i++)
        for (int c = 0; c < 5; c++) {
            const int32_t n = rd(i * 5 + c);
            ok &= (n >= 0 && n <= 7);
            const uint32_t b = (uint32_t)(i + 1 + 6 * c), v = (uint32_t)n;
            g.pl0 |= (v & 1u) << b; g.pl1 |= ((v >> 1) & 1u) << b; g.pl2 |= ((v >> 2) & 1u) << b;
        }
    for (int c = 0; c < 5; c++) {
        const int32_t n = rd(25 + c);
        ok &= (n >= 0 && n <= 15);
        const uint32_t b = (uint32_t)(6 * c), v = (uint32_t)n;
        g.pl0 |= (v & 1u) << b; g.pl1 |= ((v >> 1) & 1u) << b; g.pl2 |= ((v >> 2) & 1u) << b;
        g.pl3 |= ((v >> 3) & 1u) << b;
    }
    { const int32_t t = rd(30); ok &= (t == 0 || t == 1); g.misc |= (uint32_t)(t & 1) << 5; }
    const int o_pat = 31, o_wall = 31 + 25 * P, o_fl = 31 + 50 * P, o_sc = 31 + 51 * P, o_s = 31 + 52 * P;
    for (int p = 0; p < P; p++) {
        uint32_t pat = 0, wall = 0;
        for (int r = 0; r < 5; r++) {
            int colours = 0;
            for (int c = 0; c < 5; c++) {
                const int32_t n = rd(o_pat + 25 * p + 5 * r + c);
                ok &= (n >= 0 && n <= 7);
                if (n != 0) { colours++; pat |= ((uint32_t)c | ((uint32_t)n << 3)) << (6 * r); }
                if (rd(o_wall + 25 * p + 5 * r + c) != 0) wall |= 1u << (5 * r + c);
            }
            if (colours > 1) { ok = false; pat &= ~(63u << (6 * r)); }
        }
        const int32_t fl = rd(o_fl + p), sc = rd(o_sc + p);
        ok &= (fl >= 0 && fl <= 7 && sc >= 0 && sc <= 0xFFFF);
        g.pat[p] = pat; g.wall[p] = wall;
        g.scf[p] = ((uint32_t)sc & 0xFFFFu) | (((uint32_t)fl & 7u) << 16);
        const int32_t fps = rd(o_s + 15 + p), fpen = -rd(o_s + 15 + P + p), mc = rd(o_s + 15 + 2 * P + p);
        ok &= (fps >= 0 && fps <= 0xFFF && fpen >= 0 && fpen <= 0xFFFF && mc >= 0 && mc <= 15);
        g.sta[p] = ((uint32_t)fps & 0xFFFu) | (((uint32_t)fpen & 0xFFFFu) << 12) | (((uint32_t)mc & 15u) << 28);
        const int32_t cr = rd(o_s + 15 + 3 * P + 3 * p), cc = rd(o_s + 15 + 3 * P + 3 * p + 1),
                      ck = rd(o_s + 15 + 3 * P + 3 * p + 2);
        ok &= (cr >= 0 && cr <= 255 && cc >= 0 && cc <= 255 && ck >= 0 && ck <= 255);
        g.stb[p] = ((uint32_t)cr & 255u) | (((uint32_t)cc & 255u) << 8) | (((uint32_t)ck & 255u) << 16);
    }
    const int32_t cur = rd(o_s + 0), nf = rd(o_s + 1), eog = rd(o_s + 3), turn = rd(o_s + 4);
    ok &= (cur >= 0 && cur <= P && nf >= 0 && nf <= P && turn >= 0 && turn <= 0xFFF && rd(o_s + 2) == P);
    g.misc |= ((uint32_t)cur & 7u) << 6 | ((uint32_t)nf & 7u) << 9 | (eog ? 1u << 12 : 0u) | ((uint32_t)turn & 0xFFFu) << 16;
    for (int c = 0; c < 5; c++) {
        const int32_t b = rd(o_s + 5 + c), l = rd(o_s + 10 + c);
        ok &= (b >= 0 && b <= 63 && l >= 0 && l <= 63);
        g.box |= ((uint32_t)b & 63u) << (6 * c); g.lid |= ((uint32_t)l & 63u) << (6 * c);
    }
    g.steps = (uint32_t)rd(o_s + 15 + 6 * P);
    g.add_status((uint32_t)rd(o_s + 16 + 6 * P) & (ST_STUCK | ST_BAG_EMPTY | ST_BAD_IMPORT));
    if (!ok) g.add_status(ST_BAD_IMPORT);
    return ok;
}

template <int P, typename Wr>
AZB_HD void export_record(const Game<P>& g, Wr wr)
{
    for (int i = 0; i < 5; i++)
        for (int c = 0; c < 5; c++) {
            const uint32_t b = (uint32_t)(i + 1 + 6 * c);
            wr(i * 5 + c, (int32_t)(((g.pl0 >> b) & 1u) | (((g.pl1 >> b) & 1u) << 1) | (((g.pl2 >> b) & 1u) << 2)));
        }
    for (int c = 0; c < 5; c++) {
        const uint32_t b = (uint32_t)(6 * c);
        wr(25 + c, (int32_t)(((g.pl0 >> b) & 1u) | (((g.pl1 >> b) & 1u) << 1) | (((g.pl2 >> b) & 1u) << 2) |
                             (((g.pl3 >> b) & 1u) << 3)));
    }
    wr(30, (int32_t)((g.misc >> 5) & 1u));
    const int o_pat = 31, o_wall = 31 + 25 * P, o_fl = 31 + 50 * P, o_sc = 31 + 51 * P, o_s = 31 + 52 * P;
    for (int p = 0; p < P; p++) {
        for (int r = 0; r < 5; r++) {
            const uint32_t cnt = (g.pat[p] >> (6 * r + 3)) & 7u, col = (g.pat[p] >> (6 * r)) & 7u;
            for (int c = 0; c < 5; c++) {
                wr(o_pat + 25 * p + 5 * r + c, (int32_t)((cnt && col == (uint32_t)c) ? cnt : 0u));
                wr(o_wall + 25 * p + 5 * r + c, (int32_t)((g.wall[p] >> (5 * r + c)) & 1u));
            }
        }
        wr(o_fl + p, (int32_t)((g.scf[p] >> 16) & 7u));
        wr(o_sc + p, (int32_t)(g.scf[p] & 0xFFFFu));
        wr(o_s + 15 + p, (int32_t)(g.sta[p] & 0xFFFu));
        wr(o_s + 15 + P + p, -(int32_t)((g.sta[p] >> 12) & 0xFFFFu));
        wr(o_s + 15 + 2 * P + p, (int32_t)(g.sta[p] >> 28));
        wr(o_s + 15 + 3 * P + 3 * p + 0, (int32_t)(g.stb[p] & 255u));
        wr(o_s + 15 + 3 * P + 3 * p + 1, (int32_t)((g.stb[p] >> 8) & 255u));
        wr(o_s + 15 + 3 * P + 3 * p + 2, (int32_t)((g.stb[p] >> 16) & 255u));
    }
    wr(o_s + 0, (int32_t)g.current_player());
    wr(o_s + 1, (int32_t)g.next_first_player());
    wr(o_s + 2, P);
    wr(o_s + 3, (int32_t)g.ended());
    wr(o_s + 4, (int32_t)g.turn_counter());
    for (int c = 0; c < 5; c++) {
        wr(o_s + 5 + c, (int32_t)((g.box >> (6 * c)) & 63u));
        wr(o_s + 10 + c, (int32_t)((g.lid >> (6 * c)) & 63u));
    }
    wr(o_s + 15 + 6 * P, (int32_t)g.steps);
    wr(o_s + 16 + 6 * P, (int32_t)g.status());
}

// ---- K-step random-agent rollout of one slot (kernel K1+K2+K3+K6 body) ---------------------
// counters (DESIGN.md "rollout counters"): 0 steps, 1 games finished, 2 rounds started,
// 3 sum score seat 0, 4 sum score seat 1, 5 games seat 0 won, 6 stuck aborts, 7 games that ran the
// bag empty, 8 sum turn_counter, 9 sum -floor_penalty seat 0, 10 sum max_combo seat 0, 11 completed
// rows, 12 completed columns, 13 completed colours (seat 0), 14 sum first_player_stats seat 0,
// 15 sum of all seats' scores.  Sink::add_group(index, value) receives a lane's increments and may aggregate
// those of all lanes (the rollout kernel keeps them in registers and reduces them with one REDUX per counter and warp
// every 256 end-of-round passes: Sink::pass_done() is called by the whole group after each pass); rollout_steps
// hands its per-call totals of steps and rounds to Sink::add(index, value), called by the whole group.
// `fin` selects the games of the calling group that just ended.
template <class GT, typename Sink>
AZB_HD void tally_finished(const GT& g, Sink& sink, bool fin = true)
{
    const uint32_t s0 = g.scf[0] & 0xFFFFu, s1 = g.scf[1] & 0xFFFFu, f = fin ? 1u : 0u;
    uint32_t all = 0;
#pragma unroll
    for (int p = 0; p < GT::PLAYERS; p++) all += g.scf[p] & 0xFFFFu;
    sink.add_group(1, f);
    sink.add_group(3, f * s0);
    sink.add_group(4, f * s1);
    sink.add_group(5, f * (s0 > s1 ? 1u : 0u));
    sink.add_group(8, f * g.turn_counter());
    sink.add_group(9, f * ((g.sta[0] >> 12) & 0xFFFFu));
    sink.add_group(10, f * (g.sta[0] >> 28));
    sink.add_group(11, f * (g.stb[0] & 255u));
    sink.add_group(12, f * ((g.stb[0] >> 16) & 255u));
    sink.add_group(13, f * ((g.stb[0] >> 8) & 255u));
    sink.add_group(14, f * (g.sta[0] & 0xFFFu));
    sink.add_group(15, f * all);
}

// Where the random agent's action words come from.  The word of env step T of a slot is always
// Philox(gid, T >> 2, ACTION, 0)[T & 3]; the policies differ in WHEN the Philox blocks are computed.
// InlineWords computes a block when a game first needs it (every fourth step of each game, at a
// different time for every lane of a warp).
struct InlineWords {
    uint32_t w[4];
    uint32_t block;
    bool have;
    AZB_M InlineWords() : block(0u), have(false) { w[0] = w[1] = w[2] = w[3] = 0u; }
    AZB_M void prefetch(const Philox&, uint32_t, uint32_t) {}
    AZB_M uint32_t get(const Philox& rng, uint32_t gid, uint32_t T)
    {
        if (!have || block != (T >> 2)) { block = T >> 2; rng(gid, block, PURPOSE_ACTION, 0u, w); have = true; }
        const uint32_t i = T & 3u;
        return i == 0u ? w[0] : i == 1u ? w[1] : i == 2u ? w[2] : w[3];
    }
};

// Warp-vote policies for rollout_steps: the kernels vote across the 32 games of a warp, the host
// harness (one game at a time) votes with itself.
struct SingleLane {
    static constexpr int LANES = 1;
    AZB_M int count(bool p) const { return p ? 1 : 0; }
};
#if defined(__CUDACC__)
struct WarpLanes {
    static constexpr int LANES = 32;
    __device__ __forceinline__ int count(bool p) const { return __popc(__ballot_sync(0xFFFFFFFFu, p)); }
};
#endif

// Each slot executes exactly k_steps env steps.  A step is split in two phases so that a warp
// does not pay for the rare, long end-of-round work on every iteration:
//   light  legal mask -> random action -> move (azul.py:304) -> next_player, every iteration;
//   heavy  count_score -> end_of_game ? tally + fresh game : new_round (azul.py:306-311), run by the
//          warp only once `defer` of its games are waiting for it (or nothing else can move).
// A game that finished its round simply waits for the next heavy pass; its trajectory, and so every
// result, is independent of `defer` and of which games share its warp.
// TURNS (the rotating rollout kernel, k_rollout_rotate): the group stops right after its `max_passes`-th end-of-round pass --
// every game is then between two moves -- and the steps each game still has to take are returned; the caller continues
// them with another call (k_steps = the returned count: a trajectory does not depend on where it is cut).  Otherwise the
// call runs to the end and returns 0.
template <int P, int POOL, bool TURNS = false, typename Sink, typename Vote, typename Words>
AZB_HD int rollout_steps(Game<P>& g, const Philox& rng, uint32_t gid, int first_rule, int k_steps, Sink& sink,
                         const Vote vote, bool valid, int defer, Words& words, int max_passes = 0)
{
    uint32_t rounds = 0;
    int n_pass = 0;
    int remaining = valid ? k_steps : 0;
    // 0 playing, 1 round over: waits for score + refill, 2 waits for a fresh game (stuck / ended on entry)
    int phase = (remaining > 0 && g.ended()) ? 2 : 0;
    words.prefetch(rng, gid, g.steps);
    const bool partial = defer < Vote::LANES;                         // passes may start before every lane waits
    uint32_t open[P];                                                 // open_rows of every player, kept current
#pragma unroll
    for (int p = 0; p < P; p++) open[p] = open_rows(g, p);
    for (;;) {
        if (remaining > 0 && phase == 0) {
            uint32_t m[6];
            legal_mask_open(g, open, m);
            if (m[0] == 0u) {                                         // words 1..5 are subsets of word 0 (the floor takes any source)
                sink.add_group(6, 1);                                 // stuck round (SURVEY §5): abort the game
                phase = 2;
            } else {
                uint32_t mp, mb;
                random_action_pb(m, words.get(rng, gid, g.steps), mp, mb);   // m[0] != 0: an action exists
                apply_move_core<P, POOL, true>(g, mp, mb, open);          // azul.py:304
                g.steps += 1u;
                remaining--;
                if (is_end_of_round(g)) phase = 1;                    // azul.py:306
                else next_player(g);                                  // azul.py:313
            }
        }
        const int n_movable = vote.count(remaining > 0 && phase == 0);
        // with defer = all lanes (the default) a pass can only be due when nothing can move: one vote per light step
        const int n_waiting = (n_movable == 0 || partial) ? vote.count(phase != 0) : 0;
        if (n_waiting > 0 && (n_waiting >= defer || n_movable == 0)) {
            if (phase != 0) {
                bool fresh = phase == 2;
                phase = 0;
                rounds++;
                bool over = false;
                if (!fresh) {
                    count_score<P, POOL>(g);                          // azul.py:307
                    over = is_end_of_game(g);                         // azul.py:308-309
                    if (over) g.misc |= 1u << 12;
                }
                tally_finished(g, sink, over);                        // every waiting game calls it: one aggregated add
                fresh = fresh || over;
                uint32_t purpose = PURPOSE_REFILL;
                if (fresh) {                                          // Azul(rules), game_runner.py:79
                    uint32_t first = (uint32_t)first_rule;
                    if (first_rule == 0) {                            // azul.py:36-37 random.choice
                        uint32_t w[4];
                        rng(gid, g.steps, PURPOSE_FIRST, 0u, w);
                        first = 1u + mulhi(w[0], (uint32_t)P);
                    }
                    init_game<P, POOL>(g, first);
                    purpose = PURPOSE_RESET_REFILL;
                }
                const uint32_t bag_before = g.status() & ST_BAG_EMPTY;
                new_round_philox<P, POOL>(g, rng, gid, purpose);      // azul.py:311 / game_runner.py:80
                if (!bag_before && (g.status() & ST_BAG_EMPTY)) sink.add_group(7, 1);
#pragma unroll
                for (int p = 0; p < P; p++) open[p] = open_rows(g, p);   // scoring emptied lines and filled the wall
                words.prefetch(rng, gid, g.steps);                    // the whole warp is here: words for the next round
            }
            sink.pass_done();                                         // every lane of the group is here
            if (TURNS && ++n_pass >= max_passes) break;
        } else if (n_movable == 0) {
            break;
        }
    }
    sink.add(0, valid ? (uint32_t)(k_steps - remaining) : 0u);        // the whole group is here
    sink.add(2, valid ? rounds : 0u);
    return remaining;
}

// ---- GameRunner.step's opponent loop + reward (game_runner.py:46-52), random-agent opponent ----
// Plays random-agent moves (Philox ACTION words, like the rollout) until it is seat 1's turn with at
// least two legal actions (require_two: the reference also lets the opponent agent play seat 1's
// forced moves, game_runner.py:46; GameRunner.reset does not, :84-85) or the game is over.  Returns
// the score difference seat 1 - seat 2 after a count_score on a copy (game_runner.py:48-50).  GREEDY: the greedy agent
// (greedy_action) picks the opponent's moves from the same words.
template <int P, int POOL, bool GREEDY = false>
AZB_HD int32_t opponent_random(Game<P>& g, const Philox& rng, uint32_t gid, bool require_two, uint32_t m[6])
{
    AZB_ROLLED
    for (;;) {
        legal_mask(g, m);
        if (g.ended()) break;
        const int n_valid = popc(m[0]) + popc(m[1]) + popc(m[2]) + popc(m[3]) + popc(m[4]) + popc(m[5]);
        if (g.current_player() == 1u && (!require_two || n_valid >= 2)) break;
        if (n_valid == 0) { g.add_status(ST_STUCK); break; }
        uint32_t w[4];
        rng(gid, g.steps >> 2, PURPOSE_ACTION, 0u, w);
        const uint32_t idx = g.steps & 3u;
        const uint32_t word = idx == 0u ? w[0] : idx == 1u ? w[1] : idx == 2u ? w[2] : w[3];
        advance<P, POOL>(g, opponent_pick<P, POOL, GREEDY>(g, m, word),
                         [&](Game<P>& gg) { new_round_philox<P, POOL>(gg, rng, gid, PURPOSE_REFILL); });
    }
    Game<P> cp = g;
    count_score<P, POOL>(cp);
    return (int32_t)(cp.scf[0] & 0xFFFFu) - (int32_t)(cp.scf[1] & 0xFFFFu);
}

// GameRunner.step's opponent loop + reward with the greedy agent as the opponent (the loop rule and the return value of
// opponent_random)
template <int P, int POOL>
AZB_HD int32_t opponent_greedy(Game<P>& g, const Philox& rng, uint32_t gid, bool require_two, uint32_t m[6])
{
    return opponent_random<P, POOL, true>(g, rng, gid, require_two, m);
}

}  // namespace azb
