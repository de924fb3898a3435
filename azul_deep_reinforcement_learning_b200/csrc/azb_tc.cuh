// azb_tc.cuh -- pieces shared by the tensor-core kernels (azb_policy.cu: the fused policy step; azb_update.cu: the
// Agent.update forward / backward): tile geometry and the shared-memory weight image, tcgen05 / TMEM / bulk-copy PTX
// wrappers (the mbarrier ones are in azb_mbar.cuh), the in-kernel observation builder (game_runner.py:56-72).  Device only.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

#include "azb_mbar.cuh"
#include "azb_rules.cuh"

using namespace azb;

namespace pol {

constexpr int TILE_M = 128;                 // games per tile (rows of the MMA)
constexpr int PARTS = 4;                    // threads per game: each handles 48 of the 192 epilogue columns
constexpr int THREADS = TILE_M * PARTS;
constexpr int PART_COLS = 48;
constexpr int K1 = 144, K1_CHUNKS = K1 / 8; // obs 136 -> 144 (multiple of the MMA K = 16)
constexpr int N1A = 192, N1C = 176;         // the two layer-1 MMA N blocks (rows 0..191 and 192..367 of W1)
constexpr int N1 = N1A + N1C, N1_GROUPS = N1 / 8;
constexpr int K2 = 192, K2_CHUNKS = K2 / 8;
constexpr int N2 = 192, N2_GROUPS = N2 / 8;
constexpr int M_GROUPS = TILE_M / 8;
constexpr int HID = 180, ACT = 180, OBS = 136;

// shared-memory image (bytes).  A core matrix is 8 rows x 16 bytes = 128 contiguous bytes; a tile is
// stored [k-chunk][row-group][8 rows][8 halves], so SBO (next row group) = 128 B and LBO (next k-chunk)
// = groups * 128 B.
constexpr int W1_BYTES = K1_CHUNKS * N1_GROUPS * 128;        // 105,984
constexpr int W2_BYTES = K2_CHUNKS * N2_GROUPS * 128;        //  73,728
constexpr int A_BYTES = K2_CHUNKS * M_GROUPS * 128;          //  49,152 (layer-2 A; layer-1 A aliases its start)
constexpr int OFF_W1 = 0;
constexpr int OFF_W2 = OFF_W1 + W1_BYTES;
constexpr int OFF_VEC = OFF_W2 + W2_BYTES;                    // fp32 vectors: w2c[192] b2c[1] pad[3]
constexpr int VEC_FLOATS = 192 + 4;
constexpr int PACKED_BYTES = OFF_VEC + VEC_FLOATS * 4;        // what azb_policy_pack_weights produces
constexpr int OFF_A = (PACKED_BYTES + 127) / 128 * 128;
constexpr int OFF_BAR = OFF_A + A_BYTES;                      // 2 MMA mbarriers, tmem base (+16), weight-copy mbarrier (+24)
static_assert(PACKED_BYTES % 16 == 0, "the weight image is moved with 16-byte-granular bulk copies");
constexpr int SMEM_BYTES = OFF_BAR + 32;
static_assert(SMEM_BYTES <= 232448, "policy kernel exceeds the 227 KB shared memory of an SM");

constexpr int V_W2C = 0, V_B2C = 192;
static_assert(OFF_VEC % 16 == 0 && V_W2C % 4 == 0, "vectors must allow 128-bit loads");
// The biases ride in the MMAs: the observation carries two constant-one inputs (columns OBS, OBS + 1 of the zero
// padding) whose W1 rows hold the fp16 high and low halves of b1 (22 significand bits), and the
// hidden tile carries two constant-one units (columns HID, HID + 1) whose W2 rows hold the halves of b2_actor.
constexpr int BIAS_K1 = OBS, BIAS_K2 = HID;
static_assert(BIAS_K1 + 2 <= K1 && BIAS_K2 + 2 <= K2, "no padding column left for the bias inputs");

// Where the critic's hidden units sit among the layer-1 outputs (TMEM columns HID + j, j = 0..187): units 176..179 first,
// eight empty columns, then units 0..175 from column HID + 12 = 192 on.  Layer 2 (and the update kernel's dH GEMM) write
// columns [0,192); with this order all but four critic units stay readable in TMEM after those MMAs.
constexpr int CRITIC_SHIFT = 12;
__host__ __device__ constexpr int critic_unit(int j) { return j < 4 ? 176 + j : (j < CRITIC_SHIFT || j >= CRITIC_SHIFT + 176 ? -1 : j - CRITIC_SHIFT); }

constexpr uint32_t TMEM_COLS = 512;

// ---- PTX wrappers --------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, no swizzle (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// [13:0] start >> 4, [29:16] leading byte offset >> 4 (next k-chunk), [45:32] stride byte offset >> 4 (next
// 8-row group), [47:46] version = 1, [63:61] layout type 0
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes)
{
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor (InstrDescriptor): fp32 accumulate ([5:4] = 1), fp16 x fp16 (a_format [9:7] = b_format [12:10] = 0), both K-major, M = 128
__host__ __device__ constexpr uint32_t instr_desc(int n)
{
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// the same MMA with the A operand in tensor memory (row = TMEM lane, two consecutive K elements per 32-bit column: a K = 16
// step is 8 columns); B from shared memory
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32])
{
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    tc_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
// 16 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16])
{
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
    tc_wait_ld();
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
// 16 consecutive 32-bit columns of this thread's TMEM lane <- registers (complete when tc_wait_st() returns)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
          "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
          "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
          "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Operand format of both MMAs: IEEE half (fp16), fp32 accumulation.  kind::f16 takes fp16 or bf16 at the same rate; fp16's 11-bit
// significand keeps the logits within 1e-3 of the fp32 network (bf16: 4e-3), and nothing here comes near its range: observations
// are counts <= 255 (exact), weights are O(1), and the hidden activations saturate at 65504 instead of overflowing.
__device__ __forceinline__ uint32_t pack_f16(float lo, float hi)
{
    __half2 p = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&p);
}
// 2^x on the SFU (flush-to-zero: no denormal fix-up code around it); exp(a - b) = ex2(fma(a, LOG2E, -b * LOG2E))
__device__ __forceinline__ float ex2f(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
// log2(x) on the SFU
__device__ __forceinline__ float lg2f(float x)
{
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// relu + round-to-nearest fp16 (saturating at the largest finite value) + pack of two floats in ONE instruction
__device__ __forceinline__ uint32_t pack_relu_f16(float lo, float hi)
{
    uint32_t d;
    asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// exact float of a small non-negative integer without the conversion pipe
__device__ __forceinline__ float small_int_to_float(uint32_t n) { return __uint_as_float(0x4B000000u | n) - 8388608.0f; }

// ---- observation (game_runner.py:56-72), perspective = the seat to move -----------------------
template <int IDX>
__device__ __forceinline__ float obs_value(const Game<2>& g, uint32_t pat_me, uint32_t pat_ot, uint32_t wall_me,
                                           uint32_t wall_ot, uint32_t scf_me, uint32_t scf_ot, int persp)
{
    if constexpr (IDX < 25) {                         // displays[i][c]
        constexpr int i = IDX / 5, c = IDX % 5, b = i + 1 + 6 * c;
        return small_int_to_float(((g.pl0 >> b) & 1u) | (((g.pl1 >> b) & 1u) << 1) | (((g.pl2 >> b) & 1u) << 2));
    } else if constexpr (IDX < 30) {                  // centre colour counts
        constexpr int c = IDX - 25, b = 6 * c;
        return small_int_to_float(((g.pl0 >> b) & 1u) | (((g.pl1 >> b) & 1u) << 1) | (((g.pl2 >> b) & 1u) << 2) |
                                  (((g.pl3 >> b) & 1u) << 3));
    } else if constexpr (IDX == 30) {                 // first-player token
        return (g.misc & 32u) ? 1.0f : 0.0f;
    } else if constexpr (IDX < 81) {                  // pattern lines, mine then the opponent's
        constexpr int q = IDX - 31, r = (q % 25) / 5, c = q % 5;
        const uint32_t pat = q < 25 ? pat_me : pat_ot;
        const uint32_t cnt = (pat >> (6 * r + 3)) & 7u, col = (pat >> (6 * r)) & 7u;
        // integer select, then ONE unconditional conversion: `cond ? convert(cnt) : 0.0f` compiles to a branch per entry
        return small_int_to_float(cnt & (0u - (uint32_t)(col == (uint32_t)c)));
    } else if constexpr (IDX < 131) {                 // walls (colour-indexed, game_runner.py:69)
        constexpr int q = IDX - 81, bit = q % 25;
        const uint32_t w = q < 25 ? wall_me : wall_ot;
        return ((w >> bit) & 1u) ? 1.0f : 0.0f;
    } else if constexpr (IDX == 131) { return small_int_to_float((scf_me >> 16) & 7u);
    } else if constexpr (IDX == 132) { return small_int_to_float((scf_ot >> 16) & 7u);
    } else if constexpr (IDX == 133) { return small_int_to_float(scf_me & 0xFFFFu);
    } else if constexpr (IDX == 134) { return small_int_to_float(scf_ot & 0xFFFFu);
    } else if constexpr (IDX == 135) {                // next first player seen from this seat (game_runner.py:58-61)
        const int nf = (int)g.next_first_player();
        return nf > 0 ? small_int_to_float((uint32_t)(((nf - 1 - persp) & 1) + 1)) : 0.0f;
    } else if constexpr (IDX == BIAS_K1 || IDX == BIAS_K1 + 1) {
        return 1.0f;                                  // bias inputs (see BIAS_K1)
    } else {
        return 0.0f;
    }
}

template <int CH, int STRIDE>
__device__ __forceinline__ void obs_chunks(const Game<2>& g, uint32_t pat_me, uint32_t pat_ot, uint32_t wall_me,
                                           uint32_t wall_ot, uint32_t scf_me, uint32_t scf_ot, int persp,
                                           unsigned char* a_tile, int row)
{
    if constexpr (CH < K1_CHUNKS) {
#define OV(i) obs_value<8 * CH + (i)>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp)
        uint4 v;
        v.x = pack_f16(OV(0), OV(1)); v.y = pack_f16(OV(2), OV(3));
        v.z = pack_f16(OV(4), OV(5)); v.w = pack_f16(OV(6), OV(7));
#undef OV
        *reinterpret_cast<uint4*>(a_tile + (CH * M_GROUPS + (row >> 3)) * 128 + (row & 7) * 16) = v;
        obs_chunks<CH + STRIDE, STRIDE>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row);
    }
}

// the four threads of a game build the 18 observation chunks round-robin (part is warp-uniform)
__device__ __forceinline__ void build_obs_tile(const Game<2>& g, unsigned char* a_tile, int row, int part)
{
    const int persp = g.seat();
    const uint32_t pat_me = g.sel(g.pat, persp), pat_ot = g.sel(g.pat, 1 - persp);
    const uint32_t wall_me = g.sel(g.wall, persp), wall_ot = g.sel(g.wall, 1 - persp);
    const uint32_t scf_me = g.sel(g.scf, persp), scf_ot = g.sel(g.scf, 1 - persp);
    switch (part) {
    case 0: obs_chunks<0, PARTS>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    case 1: obs_chunks<1, PARTS>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    case 2: obs_chunks<2, PARTS>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    default: obs_chunks<3, PARTS>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    }
}

// parts 1..3 build the NEXT tile's observation (6 chunks each) while part 0 plays this tile's moves
__device__ __forceinline__ void build_obs_tile_3(const Game<2>& g, unsigned char* a_tile, int row, int part)
{
    const int persp = g.seat();
    const uint32_t pat_me = g.sel(g.pat, persp), pat_ot = g.sel(g.pat, 1 - persp);
    const uint32_t wall_me = g.sel(g.wall, persp), wall_ot = g.sel(g.wall, 1 - persp);
    const uint32_t scf_me = g.sel(g.scf, persp), scf_ot = g.sel(g.scf, 1 - persp);
    switch (part) {
    case 1: obs_chunks<0, 3>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    case 2: obs_chunks<1, 3>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    default: obs_chunks<2, 3>(g, pat_me, pat_ot, wall_me, wall_ot, scf_me, scf_ot, persp, a_tile, row); break;
    }
}

// 6 x 30-bit mask words (word p = destination p) -> 180 contiguous bits, bit a = action a
__device__ __forceinline__ void linear_mask(const uint32_t m[6], uint32_t lin[6])
{
    lin[0] = m[0] | (m[1] << 30);
    lin[1] = (m[1] >> 2) | (m[2] << 28);
    lin[2] = (m[2] >> 4) | (m[3] << 26);
    lin[3] = (m[3] >> 6) | (m[4] << 24);
    lin[4] = (m[4] >> 8) | (m[5] << 22);
    lin[5] = m[5] >> 10;
}

// 16 consecutive fp32 constants (bias / weight vectors in shared memory; 16-byte aligned by construction)
__device__ __forceinline__ void ld16f(const float* p, float (&b)[16])
{
    const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const float4 t = q[i];
        b[4 * i] = t.x; b[4 * i + 1] = t.y; b[4 * i + 2] = t.z; b[4 * i + 3] = t.w;
    }
}

__device__ __forceinline__ uint32_t pick6(const uint32_t (&a)[6], int i)
{
    return i == 0 ? a[0] : i == 1 ? a[1] : i == 2 ? a[2] : i == 3 ? a[3] : i == 4 ? a[4] : a[5];
}

}  // namespace pol
