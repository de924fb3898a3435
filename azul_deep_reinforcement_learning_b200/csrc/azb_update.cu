// azb_update.cu -- Agent.update (reference azulnet/agent.py:39-62) on the tensor cores: forward recomputation of
// ActorCritic (model.py:23-41) on the recorded decisions, the loss of agent.py:45-56 with the per-decision terms of
// nn_runner.py:32-40, and the gradient with respect to all eight parameter tensors -- hand-written tcgen05 kernels, no
// library GEMM and no autograd.
//
// Two kernels:
//   k_update_fwd_bwd  one persistent CTA per SM, 128 decisions per tile, same geometry as the policy kernel (azb_policy.cu):
//       X   = observation of the recorded packed state (built in-kernel, fp16, with the two constant-one bias inputs)
//       Ha  = relu(X W1a^T + b1a), Hc = relu(X W1c^T + b1c)                 layer 1: tcgen05.mma -> TMEM [0,368)
//       L   = Ha W2a^T + b2a                                               layer 2: tcgen05.mma -> TMEM [0,192)
//       masked log-softmax, value = Hc.w2c + b2c, log pi(a), entropy term, advantage, the three loss sums
//       dL  = d loss / d logits (per row, on CUDA cores),  dv = d loss / d value
//       dHa = (dL W2a) * (Ha > 0)                                          tcgen05.mma (W2 image as an MN-major B operand)
//       dHc = dv w2c * (Hc > 0);  grad w2c += dv Hc;  grad b2c += dv        CUDA cores
//     and writes the operand tiles X, Ha, dL, dHa, dHc (fp16, in the shared-memory core-matrix layout) to HBM.
//   k_update_dw       dW = A^T B summed over all tiles, both operands MN-major straight from those tiles (bulk-copied
//     into a four-stage shared-memory ring of half tiles), accumulators in TMEM for the whole kernel; the three products
//     run side by side in one launch (CTA b works on product b % 3):
//       grad W2a | b2a = dL^T  [Ha | 1]      grad W1a | b1a = dHa^T [X | 1]      grad W1c | b1c = dHc^T [X | 1]
//     (the bias gradients are the columns of the constant-one inputs), reduced into the global gradient with atomics.
// Gradients are SUMS over the decisions (the caller divides by the global decision count after the all-reduce).
// Operands are fp16 (11-bit significands), accumulation is fp32.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "azb_internal.h"
#include "azb_rules.cuh"
#include "azb_tc.cuh"

namespace upd {

using namespace pol;

constexpr int X_TILE_BYTES = K1_CHUNKS * M_GROUPS * 128;     // 36,864: [18 chunks][16 row groups][8 rows][8 halves]
constexpr int H_TILE_BYTES = A_BYTES;                        // 49,152: [24 chunks][16 row groups][8 rows][8 halves]
constexpr int CHUNKS_PER_PART = PART_COLS / 8;               // 6
// In HBM a tile is stored as two halves of 64 decisions, each [column chunk][8 row groups][8 rows][8 halves] and
// contiguous, so that k_update_dw can stream half tiles (a four-stage ring instead of two stages of whole tiles).
__device__ __forceinline__ int hbm_off(int chunk, int row, int chunks)
{
    return (((row >> 6) * chunks + chunk) * 8 + ((row >> 3) & 7)) * 128 + (row & 7) * 16;
}

struct FwdArgs {
    const uint32_t* __restrict__ state_rec;   // [17][cap] packed states the decisions were taken on
    int64_t cap;
    const uint8_t* __restrict__ action;       // [cap]
    const float* __restrict__ qval;           // [cap] discounted returns
    const uint32_t* __restrict__ n_dec;       // [1] device-side decision count (clamped to cap), or null: n_fixed
    int64_t n_fixed;
    int64_t row0, rows_max;                   // this launch handles decisions [row0, row0 + rows_max) (workspace-sized chunks)
    const unsigned char* __restrict__ packed; // weight image (azb_policy_pack_weights)
    float actor_c, critic_c, entropy_c;
    unsigned char* __restrict__ xt;           // operand tiles for k_update_dw, [tiles][...]
    unsigned char* __restrict__ ha;
    unsigned char* __restrict__ dl;
    unsigned char* __restrict__ dha;
    unsigned char* __restrict__ dhc;
    float* __restrict__ grad_w2c;             // [180] +=   critic_linear2.weight
    float* __restrict__ grad_b2c;             // [1]   +=   critic_linear2.bias
    double* __restrict__ sums;                // [3]   +=   sum(-log_prob * advantage), sum(advantage^2), sum(entropy term)
    float* __restrict__ logits_out;           // [n][180] optional (parity tests)
    float* __restrict__ value_out;            // [n] optional
};

__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

// scratch in the tail of the tile region (free while no MMA reads it): per (part, row) softmax / critic partials
constexpr int SCR_WORDS = 6;                                  // m, s, sl, value, n | flags, logit of the taken action
constexpr int OFF_SCR = X_TILE_BYTES;                         // [SCR_WORDS][PARTS * TILE_M] floats = 12,288 bytes: exactly the tail
static_assert(OFF_SCR + SCR_WORDS * THREADS * 4 <= A_BYTES, "scratch exceeds the tile");

__global__ void __launch_bounds__(THREADS, 1) k_update_fwd_bwd(FwdArgs A)
{
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, row = tid & (TILE_M - 1), part = tid >> 7;
    unsigned char* t1 = smem + OFF_A;
    const float* vec = reinterpret_cast<const float*>(smem + OFF_VEC);
    const uint32_t bar1 = smem_u32(smem + OFF_BAR), bar2 = bar1 + 8, bar_w = bar1 + 24;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + OFF_BAR + 16);
    float* scr = reinterpret_cast<float*>(t1 + OFF_SCR);
    __shared__ uint64_t bar3_storage;
    __shared__ double red[3][THREADS / 32];
    const uint32_t bar3 = smem_u32(&bar3_storage);

    if (tid == 0) {
        mbar_init(bar1, 1); mbar_init(bar2, 1); mbar_init(bar3, 1); mbar_init(bar_w, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_w), "r"((uint32_t)PACKED_BYTES) : "memory");
        constexpr uint32_t CHUNK = 32768;
        for (uint32_t off = 0; off < (uint32_t)PACKED_BYTES; off += CHUNK) {
            const uint32_t bytes = (uint32_t)PACKED_BYTES - off < CHUNK ? (uint32_t)PACKED_BYTES - off : CHUNK;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32(smem) + off), "l"(A.packed + off), "r"(bytes), "r"(bar_w) : "memory");
        }
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_row = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    // columns [368, 376): read by the critic chunks (180 + 191 = 371), never written by an MMA
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(tmem_row + N1), "r"(0u) : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");

    const uint32_t w1_addr = smem_u32(smem + OFF_W1), w2_addr = smem_u32(smem + OFF_W2), a_addr = smem_u32(t1);
    int64_t n_all = A.n_dec ? (int64_t)*A.n_dec : A.n_fixed;
    n_all = n_all < A.cap ? n_all : A.cap;
    int64_t n = n_all - A.row0;                              // decisions of this chunk
    n = n < 0 ? 0 : (n < A.rows_max ? n : A.rows_max);
    const int64_t tiles = (n + TILE_M - 1) / TILE_M;
    const int col0 = part * PART_COLS;
    uint32_t phase = 0;
    double acc_a = 0.0, acc_c = 0.0, acc_e = 0.0;            // loss sums (part 0 threads)
    float gw2c[3] = {0.0f, 0.0f, 0.0f}, gb2c = 0.0f;          // lane l of a warp: critic columns col0 + 16 c + (l & 15), c = 0..2

    // the packed state of a tile's decisions is loaded one tile ahead (before the previous tile's last epilogue)
    Game<2> nxt;
    if ((int64_t)blockIdx.x < tiles) {
        const int64_t g0 = (int64_t)blockIdx.x * TILE_M + row;
        nxt.load(A.state_rec, A.cap, A.row0 + (g0 < n ? g0 : n - 1));
    }
    mbar_wait(bar_w, 0);
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        const bool valid = tile * TILE_M + row < n;
        const int64_t g = A.row0 + tile * TILE_M + row;         // absolute decision index
        const int64_t gl = valid ? g : A.row0 + n - 1;
        unsigned char* g_x = A.xt + tile * X_TILE_BYTES;
        unsigned char* g_ha = A.ha + tile * H_TILE_BYTES;
        unsigned char* g_dl = A.dl + tile * H_TILE_BYTES;
        unsigned char* g_dha = A.dha + tile * H_TILE_BYTES;
        unsigned char* g_dhc = A.dhc + tile * H_TILE_BYTES;

        // ---- observation of the recorded state (mover's perspective, game_runner.py:56-72) and its legal mask ----
        uint64_t mybits;
        {
            const Game<2> gm = nxt;
            build_obs_tile(gm, t1, row, part);
            uint32_t m[6], lin[6];
            legal_mask(gm, m);
            linear_mask(m, lin);
            const int w = col0 >> 5, sh = col0 & 31;
            mybits = ((((uint64_t)pick6(lin, w + 1) << 32) | pick6(lin, w)) >> sh) & 0xFFFFFFFFFFFFull;
        }
        const int act = (int)A.action[gl];
        const float q = A.qval[gl];
        fence_async_smem();
        tc_fence_before();
        __syncthreads();

        // ---- layer 1 ----
        if (tid == 0) {
            tc_fence_after();
            // (unrolled, one add per descriptor and k-step: the start-address field never carries out of its 14 bits; see k_policy)
            const uint64_t ad0 = smem_desc(a_addr, M_GROUPS * 128, 128);
            const uint64_t ba0 = smem_desc(w1_addr, N1_GROUPS * 128, 128);
            const uint64_t bc0 = smem_desc(w1_addr + (N1A / 8) * 128, N1_GROUPS * 128, 128);
#pragma unroll
            for (int s = 0; s < K1 / 16; s++) {
                const uint64_t ad = ad0 + (uint64_t)(s * ((2 * M_GROUPS * 128) >> 4));
                const uint64_t bo = (uint64_t)(s * ((2 * N1_GROUPS * 128) >> 4));
                umma(tmem_base, ad, ba0 + bo, instr_desc(N1A), s > 0);
                umma(tmem_base + N1A, ad, bc0 + bo, instr_desc(N1C), s > 0);
            }
            umma_commit(bar1);
        }
        // the X tile goes to HBM for k_update_dw: every thread copies the chunks of its own row that it will overwrite in
        // epilogue 1 (chunks 6 * part .. + 5; X has 18), so no other thread's write can race with the copy
        if (part < 3) {
#pragma unroll
            for (int c = 0; c < CHUNKS_PER_PART; c++) {
                const int off = ((CHUNKS_PER_PART * part + c) * M_GROUPS + (row >> 3)) * 128 + (row & 7) * 16;
                *reinterpret_cast<uint4*>(g_x + hbm_off(CHUNKS_PER_PART * part + c, row, K1_CHUNKS)) = *reinterpret_cast<const uint4*>(t1 + off);
            }
        }
        mbar_wait(bar1, phase);
        tc_fence_after();

        // ---- epilogue 1: Ha -> relu -> fp16 -> shared memory (layer-2 A operand) and HBM; which units are active ----
        uint64_t hmask = 0ull;
#pragma unroll
        for (int cc = 0; cc < PART_COLS / 16; cc++) {
            const int c0 = col0 + 16 * cc;
            float v[16];
            tmem_ld16(tmem_row + c0, v);
#pragma unroll
            for (int qq = 0; qq < 2; qq++) {
                uint4 o;
                uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
                for (int e = 0; e < 4; e++) {
                    const int j = c0 + 8 * qq + 2 * e;
                    ow[e] = j < HID ? pack_relu_f16(v[8 * qq + 2 * e], v[8 * qq + 2 * e + 1]) : (j == BIAS_K2 ? 0x3C003C00u : 0u);
                }
                const int off = (((c0 >> 3) + qq) * M_GROUPS + (row >> 3)) * 128 + (row & 7) * 16;
                *reinterpret_cast<uint4*>(t1 + off) = o;
                *reinterpret_cast<uint4*>(g_ha + hbm_off((c0 >> 3) + qq, row, K2_CHUNKS)) = o;
            }
#pragma unroll
            for (int i = 0; i < 16; i++) hmask |= (uint64_t)((c0 + i < HID && v[i] > 0.0f) ? 1u : 0u) << (16 * cc + i);
        }
        // ---- critic head: partial value over this part's columns, which units are active; the four units that live in
        // columns 180..183 (overwritten by layer 2) are kept in registers by part 0 ----
        float value_p = 0.0f, save4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        uint64_t cmask = 0ull;
#pragma unroll
        for (int cc = 0; cc < PART_COLS / 16; cc++) {
            const int c0 = col0 + 16 * cc;
            float v[16], ww[16];
            tmem_ld16(tmem_row + HID + c0, v);
            ld16f(vec + V_W2C + c0, ww);
#pragma unroll
            for (int i = 0; i < 16; i++) {
                value_p = fmaf(fmaxf(v[i], 0.0f), ww[i], value_p);
                cmask |= (uint64_t)(v[i] > 0.0f ? 1u : 0u) << (16 * cc + i);
            }
            if (cc == 0) { save4[0] = v[0]; save4[1] = v[1]; save4[2] = v[2]; save4[3] = v[3]; }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();

        // ---- layer 2 ----
        if (tid == 0) {
            tc_fence_after();
            const uint64_t ad0 = smem_desc(a_addr, M_GROUPS * 128, 128), bd0 = smem_desc(w2_addr, N2_GROUPS * 128, 128);
#pragma unroll
            for (int s = 0; s < K2 / 16; s++)
                umma(tmem_base, ad0 + (uint64_t)(s * ((2 * M_GROUPS * 128) >> 4)), bd0 + (uint64_t)(s * ((2 * N2_GROUPS * 128) >> 4)),
                     instr_desc(N2), s > 0);
            umma_commit(bar2);
        }
        mbar_wait(bar2, phase);
        tc_fence_after();

        // ---- epilogue 2a: softmax statistics of this part's 48 columns (legal ones), the taken action's logit ----
        float mx = -INFINITY, se = 0.0f, sl = 0.0f, la = 0.0f;
#pragma unroll
        for (int c = 0; c < PART_COLS / 16; c++) {
            const int c0 = col0 + 16 * c;
            float v[16];
            tmem_ld16(tmem_row + c0, v);
            const uint32_t bits = (uint32_t)(mybits >> (16 * c)) & 0xFFFFu;
            if (A.logits_out && valid) {
#pragma unroll
                for (int i = 0; i < 16; i++)
                    if (c0 + i < ACT) A.logits_out[g * ACT + c0 + i] = v[i];
            }
            float cm = -INFINITY;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const bool legal = (bits >> i) & 1u;
                la = (c0 + i == act) ? v[i] : la;
                sl += legal ? v[i] : 0.0f;
                v[i] = legal ? v[i] : -INFINITY;
                cm = fmaxf(cm, v[i]);
            }
            const float nm = fmaxf(mx, cm);
            const float ms = nm == -INFINITY ? 0.0f : nm;
            float sum = 0.0f;
#pragma unroll
            for (int i = 0; i < 16; i++) sum += __expf(v[i] - ms);
            se = se * __expf(mx - ms) + sum;
            mx = nm;
        }
        {
            const int slot = part * TILE_M + row;
            // this part holds the taken action's column AND the action is legal there
            const bool owns = act >= col0 && act < col0 + PART_COLS && ((mybits >> (act - col0)) & 1ull);
            scr[0 * THREADS + slot] = mx; scr[1 * THREADS + slot] = se; scr[2 * THREADS + slot] = sl;
            scr[3 * THREADS + slot] = value_p;
            scr[4 * THREADS + slot] = __int_as_float(__popcll(mybits) | (owns ? 256 : 0));
            scr[5 * THREADS + slot] = la;
        }
        __syncthreads();

        // ---- epilogue 2b: merge the four parts of the row (all four threads compute the same numbers) ----
        float gmx = -INFINITY, gsl = 0.0f, value = vec[V_B2C], la_row = 0.0f;
        int n_valid = 0;
        bool act_seen = false;
#pragma unroll
        for (int qq = 0; qq < PARTS; qq++) {
            const int slot = qq * TILE_M + row;
            const int nf = __float_as_int(scr[4 * THREADS + slot]);
            const float pm = scr[0 * THREADS + slot];
            if ((nf & 255) > 0) gmx = fmaxf(gmx, pm);
            gsl += scr[2 * THREADS + slot]; value += scr[3 * THREADS + slot]; n_valid += nf & 255;
            if (nf & 256) { la_row = scr[5 * THREADS + slot]; act_seen = true; }
        }
        float gse = 0.0f;
#pragma unroll
        for (int qq = 0; qq < PARTS; qq++) {
            const int slot = qq * TILE_M + row;
            const int nf = __float_as_int(scr[4 * THREADS + slot]);
            if ((nf & 255) > 0) gse += scr[1 * THREADS + slot] * __expf(scr[0 * THREADS + slot] - gmx);
        }
        // rows past the end and rows whose action is not legal (no legal action at all, action >= 180, or a masked-out
        // action) contribute nothing (model.py:33-34): act_seen is set only by the part where the action is legal
        const bool ok = valid && act_seen;
        const float lse = ok ? gmx + __logf(gse) : 0.0f;
        const float log_prob = ok ? la_row - lse : 0.0f;                                   // nn_runner.py:32
        const float inv_k = ok ? 1.0f / (float)n_valid : 0.0f;
        const float entropy = ok ? -(gsl * inv_k - lse) : 0.0f;                            // nn_runner.py:36-40
        const float adv = ok ? q - value : 0.0f;                                           // agent.py:45
        // value enters through advantage in the actor AND the critic term (agent.py:45-50: advantage is not detached)
        const float dv = ok ? A.actor_c * log_prob - 2.0f * A.critic_c * adv : 0.0f;
        if (part == 0 && ok) {
            acc_a += (double)(-log_prob * adv); acc_c += (double)(adv * adv); acc_e += (double)entropy;
            if (A.value_out) A.value_out[g] = value;
        }
        __syncthreads();                                   // scratch reads are done before the dL tile overwrites that region

        // ---- epilogue 2c: dL = d loss / d logits for this part's columns -> fp16 -> shared memory (A of the dH GEMM) + HBM ----
#pragma unroll
        for (int c = 0; c < PART_COLS / 16; c++) {
            const int c0 = col0 + 16 * c;
            float v[16];
            tmem_ld16(tmem_row + c0, v);
            const uint32_t bits = ok ? (uint32_t)(mybits >> (16 * c)) & 0xFFFFu : 0u;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const float pj = __expf(v[i] - lse);
                // d(-log_prob * adv) / dl_j = -adv (delta_ja - p_j);   d entropy / dl_j = p_j - 1/k   (legal j only)
                const float gj = A.actor_c * (-adv) * ((c0 + i == act ? 1.0f : 0.0f) - pj) + A.entropy_c * (pj - inv_k);
                v[i] = ((bits >> i) & 1u) ? gj : 0.0f;
            }
#pragma unroll
            for (int qq = 0; qq < 2; qq++) {
                uint4 o;
                o.x = pack_f16(v[8 * qq + 0], v[8 * qq + 1]); o.y = pack_f16(v[8 * qq + 2], v[8 * qq + 3]);
                o.z = pack_f16(v[8 * qq + 4], v[8 * qq + 5]); o.w = pack_f16(v[8 * qq + 6], v[8 * qq + 7]);
                const int off = (((c0 >> 3) + qq) * M_GROUPS + (row >> 3)) * 128 + (row & 7) * 16;
                *reinterpret_cast<uint4*>(t1 + off) = o;
                *reinterpret_cast<uint4*>(g_dl + hbm_off((c0 >> 3) + qq, row, K2_CHUNKS)) = o;
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();

        // ---- dHa_pre = dL W2a on the tensor cores: A = the dL tile (K-major over the actions), B = the W2 image read as an
        // MN-major operand (N = hidden unit, contiguous in the image; K = action) -> TMEM [0,192) (the logits are consumed) ----
        if (tid == 0) {
            tc_fence_after();
            const uint64_t ad0 = smem_desc(a_addr, M_GROUPS * 128, 128);
            const uint64_t bd0 = smem_desc(w2_addr, 128, N2_GROUPS * 128);                       // LBO: next 8 actions, SBO: next 8 hidden units
#pragma unroll
            for (int s = 0; s < N2 / 16; s++)
                umma(tmem_base, ad0 + (uint64_t)(s * ((2 * M_GROUPS * 128) >> 4)), bd0 + (uint64_t)(s * ((2 * 128) >> 4)),
                     instr_desc(K2) | (1u << 16), s > 0);
            umma_commit(bar3);
        }
        // ---- meanwhile, the critic: dHc = dv w2c (Hc > 0) -> HBM;  grad w2c += dv relu(Hc_pre);  grad b2c += dv ----
#pragma unroll
        for (int c = 0; c < PART_COLS / 16; c++) {
            const int c0 = col0 + 16 * c;
            float v[16], ww[16];
            tmem_ld16(tmem_row + HID + c0, v);               // columns >= 192 hold Hc_pre; 180..191 were overwritten
            ld16f(vec + V_W2C + c0, ww);
            if (part == 0 && c == 0) {
#pragma unroll
                for (int i = 0; i < 12; i++) v[i] = i < 4 ? save4[i] : 0.0f;
            }
            const uint32_t bits = (uint32_t)(cmask >> (16 * c)) & 0xFFFFu;
            float d[16];
#pragma unroll
            for (int i = 0; i < 16; i++) d[i] = ((bits >> i) & 1u) ? dv * ww[i] : 0.0f;
#pragma unroll
            for (int qq = 0; qq < 2; qq++) {
                uint4 o;
                o.x = pack_f16(d[8 * qq + 0], d[8 * qq + 1]); o.y = pack_f16(d[8 * qq + 2], d[8 * qq + 3]);
                o.z = pack_f16(d[8 * qq + 4], d[8 * qq + 5]); o.w = pack_f16(d[8 * qq + 6], d[8 * qq + 7]);
                *reinterpret_cast<uint4*>(g_dhc + hbm_off((c0 >> 3) + qq, row, K2_CHUNKS)) = o;
            }
            // column sums over the warp's 32 rows by a transposing butterfly: at distance s every lane hands the half of its
            // values that its partner keeps (16 shuffles per 16 columns instead of 80); lane l ends up with column l & 15
            float t[16];
#pragma unroll
            for (int i = 0; i < 16; i++) t[i] = dv * fmaxf(v[i], 0.0f);
#pragma unroll
            for (int sft = 8; sft >= 1; sft >>= 1) {
                const bool up = (lane & sft) != 0;
#pragma unroll
                for (int i = 0; i < sft; i++) {
                    const float send = up ? t[i] : t[i + sft];
                    const float keep = up ? t[i + sft] : t[i];
                    t[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, sft);
                }
            }
            gw2c[c] += t[0] + __shfl_xor_sync(0xFFFFFFFFu, t[0], 16);
        }
        if (part == 0) gb2c += dv;
        if (tile + gridDim.x < tiles) {                    // in flight during epilogue 3
            const int64_t g2 = (tile + gridDim.x) * TILE_M + row;
            nxt.load(A.state_rec, A.cap, A.row0 + (g2 < n ? g2 : n - 1));
        }
        mbar_wait(bar3, phase);
        tc_fence_after();
        phase ^= 1;

        // ---- epilogue 3: dHa = dHa_pre * (Ha > 0) -> fp16 -> HBM ----
#pragma unroll
        for (int c = 0; c < PART_COLS / 16; c++) {
            const int c0 = col0 + 16 * c;
            float v[16];
            tmem_ld16(tmem_row + c0, v);
            const uint32_t bits = (uint32_t)(hmask >> (16 * c)) & 0xFFFFu;
#pragma unroll
            for (int i = 0; i < 16; i++) v[i] = ((bits >> i) & 1u) ? v[i] : 0.0f;
#pragma unroll
            for (int qq = 0; qq < 2; qq++) {
                uint4 o;
                o.x = pack_f16(v[8 * qq + 0], v[8 * qq + 1]); o.y = pack_f16(v[8 * qq + 2], v[8 * qq + 3]);
                o.z = pack_f16(v[8 * qq + 4], v[8 * qq + 5]); o.w = pack_f16(v[8 * qq + 6], v[8 * qq + 7]);
                *reinterpret_cast<uint4*>(g_dha + hbm_off((c0 >> 3) + qq, row, K2_CHUNKS)) = o;
            }
        }
        tc_fence_before();
        __syncthreads();                                   // TMEM and the tile region are free for the next tile
    }

    // ---- kernel end: the critic's second layer gradient and the loss sums ----
    {
        // lanes 0..15 of every warp hold the sums of critic columns col0 + 16 c + lane over the warp's rows
        if (lane < 16) {
#pragma unroll
            for (int c = 0; c < 3; c++) {
                const int u = critic_unit(col0 + 16 * c + lane);
                if (u >= 0 && gw2c[c] != 0.0f) atomicAdd(A.grad_w2c + u, gw2c[c]);
            }
        }
        const float b = warp_sum(gb2c);
        if (lane == 0 && b != 0.0f) atomicAdd(A.grad_b2c, b);
        double a0 = acc_a, a1 = acc_c, a2 = acc_e;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a0 += __shfl_xor_sync(0xFFFFFFFFu, a0, o); a1 += __shfl_xor_sync(0xFFFFFFFFu, a1, o); a2 += __shfl_xor_sync(0xFFFFFFFFu, a2, o);
        }
        if (lane == 0) { red[0][warp] = a0; red[1][warp] = a1; red[2][warp] = a2; }
        __syncthreads();
        if (tid < 3 && A.sums) {
            double t = 0.0;
            for (int w = 0; w < THREADS / 32; w++) t += red[tid][w];
            if (t != 0.0) atomicAdd(A.sums + tid, t);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// dW = sum over tiles of A_tile^T B_tile.  A tile: [128 decisions][192 columns], B tile: [128 decisions][NB columns], both
// fp16 in the core-matrix layout [column chunk][row group][8 rows][8 columns] -- i.e. MN-major operands (the M / N index is
// the contiguous one, K = the decision).  M = 192 is covered by two M = 128 MMAs (the second reads 64 columns past the A
// half tile: the B half follows it in the stage buffer, its values only reach accumulator rows >= 192, which are dropped).
// ---------------------------------------------------------------------------------------------------------------------
struct DwGemm {
    const unsigned char* __restrict__ a_tiles;   // [tiles][49152]
    const unsigned char* __restrict__ b_tiles;   // [tiles][b_bytes]
    int b_bytes, nb;                             // nb = columns of the B tile (192 or 144) = N of the MMA
    float* __restrict__ grad_w;                  // [180][ld] +=
    int ld, n_cols;                              // columns < n_cols go to grad_w[row][col]
    float* __restrict__ grad_b;                  // [180] += column bias_col
    int bias_col;
    int critic_rows;                             // 1: accumulator row j is critic unit critic_unit(j) (dHc tiles)
};
struct DwArgs {
    DwGemm gemm[3];                              // CTA b works on gemm[b % 3]: the three products run side by side
    const uint32_t* __restrict__ n_dec;
    int64_t n_fixed, cap, row0, rows_max;
};

constexpr int DW_THREADS = 256;
constexpr int DW_STAGES = 4;
constexpr int DW_HALF_A = H_TILE_BYTES / 2;                  // 24,576: half an A tile (64 decisions)
constexpr int DW_STAGE_BYTES = 2 * DW_HALF_A;                // A half + room for the larger B half

__device__ __forceinline__ void red_add_v4(float* dst, float a, float b, float c, float d)
{
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__global__ void __launch_bounds__(DW_THREADS, 1) k_update_dw(DwArgs A)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2 * DW_STAGES + 1];             // full[S], empty[S], done
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[DW_STAGES]), done = smem_u32(&bars[2 * DW_STAGES]);
    if (tid == 0) {
        for (int i = 0; i < 2 * DW_STAGES + 1; i++) mbar_init(smem_u32(&bars[i]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    int64_t n = A.n_dec ? (int64_t)*A.n_dec : A.n_fixed;
    n = (n < A.cap ? n : A.cap) - A.row0;
    n = n < 0 ? 0 : (n < A.rows_max ? n : A.rows_max);
    const int64_t tiles = (n + TILE_M - 1) / TILE_M;
    // CTA b: product b % 3, and among that product's CTAs number b / 3 of (gridDim.x - role + 2) / 3
    const int role = (int)(blockIdx.x % 3u), rank = (int)(blockIdx.x / 3u), ranks = ((int)gridDim.x - role + 2) / 3;
    const DwGemm& G = A.gemm[role];
    const int NB = G.nb;
    const int64_t my_tiles = rank < tiles ? (tiles - rank + ranks - 1) / ranks : 0;
    const int64_t my_halves = 2 * my_tiles;                  // work items: half tiles of 64 decisions

    if (tid == 0 && my_tiles > 0) {
        // producer and MMA issuer in one thread: up to DW_STAGES - 1 half tiles are in flight while the MMAs of one run
        const uint32_t idesc = instr_desc(NB) | (1u << 15) | (1u << 16);     // A and B MN-major
        const int b_half = G.b_bytes / 2;
        auto load = [&](int64_t i) {
            const int s = (int)(i % DW_STAGES);
            const int64_t t = (int64_t)rank + (i >> 1) * ranks;
            const uint32_t dst = smem_u32(smem) + s * DW_STAGE_BYTES, bar = full0 + 8 * s;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((uint32_t)(DW_HALF_A + b_half)) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(dst), "l"(G.a_tiles + t * H_TILE_BYTES + (i & 1) * DW_HALF_A), "r"((uint32_t)DW_HALF_A), "r"(bar) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(dst + DW_HALF_A), "l"(G.b_tiles + t * (int64_t)G.b_bytes + (i & 1) * b_half), "r"((uint32_t)b_half), "r"(bar) : "memory");
        };
        for (int64_t i = 0; i < DW_STAGES - 1 && i < my_halves; i++) load(i);
        for (int64_t i = 0; i < my_halves; i++) {
            const int s = (int)(i % DW_STAGES);
            const int64_t nx = i + DW_STAGES - 1;            // refill the stage the MMAs of item i - 1 read
            if (nx < my_halves) {
                if (i >= 1) mbar_wait(empty0 + 8 * (int)(nx % DW_STAGES), (uint32_t)(((i - 1) / DW_STAGES) & 1));
                load(nx);
            }
            mbar_wait(full0 + 8 * s, (uint32_t)((i / DW_STAGES) & 1));
            tc_fence_after();
            const uint32_t a_addr = smem_u32(smem) + s * DW_STAGE_BYTES, b_addr = a_addr + DW_HALF_A;
#pragma unroll 1
            for (int ks = 0; ks < 64 / 16; ks++) {
                // MN-major: SBO = next 8 columns (a chunk of the half tile: 8 row groups = 1,024 bytes), LBO = next 8 decisions (128 bytes)
                const uint64_t bd = smem_desc(b_addr + ks * 256, 128, 1024);
                const uint64_t ad0 = smem_desc(a_addr + ks * 256, 128, 1024);
                const uint64_t ad1 = smem_desc(a_addr + 16 * 1024 + ks * 256, 128, 1024);   // columns 128..255: runs 8 KB into the B half
                umma(tmem_base, ad0, bd, idesc, (i > 0 || ks > 0) ? 1u : 0u);
                umma(tmem_base + NB, ad1, bd, idesc, (i > 0 || ks > 0) ? 1u : 0u);
            }
            umma_commit(empty0 + 8 * s);
        }
        umma_commit(done);
    }
    if (my_tiles > 0) {
        mbar_wait(done, 0);
        tc_fence_after();
        // ---- epilogue: accumulator rows (TMEM lanes) = M index; warps 0-3 take M tile 0, warps 4-7 M tile 1; the sums of
        // this CTA's tiles are added to the global gradient with 16-byte vector reductions ----
        const int mt = warp >> 2;
        const int j = mt * 128 + (warp & 3) * 32 + lane;                       // accumulator row
        const int out_row = j < 192 ? (G.critic_rows ? critic_unit(j) : (j < HID ? j : -1)) : -1;
        const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(mt * NB);
#pragma unroll 1
        for (int c0 = 0; c0 < NB; c0 += 16) {
            float v[16];
            tmem_ld16(taddr + c0, v);
            if (out_row >= 0) {
                float* wrow = G.grad_w + (int64_t)out_row * G.ld;           // rows are 16-byte aligned: ld = 180 or 136
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                    const int col = c0 + i;
                    if (col + 4 <= G.n_cols) {
                        red_add_v4(wrow + col, v[i], v[i + 1], v[i + 2], v[i + 3]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            if (col + e < G.n_cols) atomicAdd(wrow + col + e, v[i + e]);
                            else if (col + e == G.bias_col) atomicAdd(G.grad_b + out_row, v[i + e]);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

}  // namespace upd

extern "C" {

// the kernels work through the decisions in chunks of at most UPDATE_CHUNK so that the workspace stays bounded (1.9 GB)
// however large the record capacity is
static int64_t UPDATE_CHUNK = (int64_t)1 << 20;

int azb_update_set_chunk_rows(int64_t rows)
{
    if (rows < pol::TILE_M || rows % pol::TILE_M) return azb_fail(AZB_E_INVALID, "chunk rows must be a positive multiple of 128%s");
    UPDATE_CHUNK = rows;
    return 0;
}

int64_t azb_update_workspace_bytes(int64_t capacity)
{
    const int64_t rows = capacity < UPDATE_CHUNK ? capacity : UPDATE_CHUNK;
    const int64_t tiles = (rows + pol::TILE_M - 1) / pol::TILE_M;
    return tiles * (int64_t)(upd::X_TILE_BYTES + 4 * upd::H_TILE_BYTES);
}

int azb_a2c_update_gradients(azb_t* h, const uint32_t* state_rec, int64_t capacity, const uint8_t* action, const float* qval,
                             const uint32_t* n_dec, int64_t n_fixed, const void* packed, float actor_coeff, float critic_coeff,
                             float entropy_coeff, void* workspace, float* grad_w1a, float* grad_b1a, float* grad_w2a,
                             float* grad_b2a, float* grad_w1c, float* grad_b1c, float* grad_w2c, float* grad_b2c, double* sums,
                             float* logits_out, float* value_out, void* stream)
{
    CHECK_HANDLE(h);
    if (!state_rec || !action || !qval || !packed || !workspace) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (!grad_w1a || !grad_b1a || !grad_w2a || !grad_b2a || !grad_w1c || !grad_b1c || !grad_w2c || !grad_b2c)
        return azb_fail(AZB_E_INVALID, "null gradient buffer%s");
    if (capacity < 1 || (!n_dec && (n_fixed < 0 || n_fixed > capacity))) return azb_fail(AZB_E_INVALID, "bad decision count / capacity%s");
    if (h->players != 2) return azb_fail(AZB_E_INVALID, "the policy network is defined for 2 players (136 inputs, agent.py:29)%s");
    if (!n_dec && n_fixed == 0) return 0;
    const int64_t chunk_rows = capacity < UPDATE_CHUNK ? capacity : UPDATE_CHUNK;
    const int64_t tiles_cap = (chunk_rows + pol::TILE_M - 1) / pol::TILE_M;
    unsigned char* ws = (unsigned char*)workspace;
    upd::FwdArgs F;
    F.state_rec = state_rec; F.cap = capacity; F.action = action; F.qval = qval; F.n_dec = n_dec; F.n_fixed = n_fixed;
    F.packed = (const unsigned char*)packed; F.actor_c = actor_coeff; F.critic_c = critic_coeff; F.entropy_c = entropy_coeff;
    // five arrays of operand tiles (one chunk's worth)
    F.dl = ws;
    F.ha = F.dl + tiles_cap * upd::H_TILE_BYTES;
    F.dha = F.ha + tiles_cap * upd::H_TILE_BYTES;
    F.dhc = F.dha + tiles_cap * upd::H_TILE_BYTES;
    F.xt = F.dhc + tiles_cap * upd::H_TILE_BYTES;
    F.grad_w2c = grad_w2c; F.grad_b2c = grad_b2c; F.sums = sums; F.logits_out = logits_out; F.value_out = value_out;
    cudaStream_t st = (cudaStream_t)stream;
    AZB_CUDA(cudaFuncSetAttribute(upd::k_update_fwd_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, pol::SMEM_BYTES));
    const int dw_smem = upd::DW_STAGES * upd::DW_STAGE_BYTES;
    AZB_CUDA(cudaFuncSetAttribute(upd::k_update_dw, cudaFuncAttributeMaxDynamicSharedMemorySize, dw_smem));
    upd::DwArgs D;
    D.n_dec = n_dec; D.n_fixed = n_fixed; D.cap = capacity;
    // grad W2a | b2a = dL^T [Ha | 1]
    D.gemm[0] = upd::DwGemm{F.dl, F.ha, upd::H_TILE_BYTES, 192, grad_w2a, pol::HID, pol::HID, grad_b2a, pol::BIAS_K2, 0};
    // grad W1a | b1a = dHa^T [X | 1]
    D.gemm[1] = upd::DwGemm{F.dha, F.xt, upd::X_TILE_BYTES, 144, grad_w1a, pol::OBS, pol::OBS, grad_b1a, pol::BIAS_K1, 0};
    // grad W1c | b1c = dHc^T [X | 1]
    D.gemm[2] = upd::DwGemm{F.dhc, F.xt, upd::X_TILE_BYTES, 144, grad_w1c, pol::OBS, pol::OBS, grad_b1c, pol::BIAS_K1, 1};
    const int dw_grid = h->sm_count < 3 ? 3 : h->sm_count;       // every product needs at least one CTA
    // with a device-side count every chunk of the capacity is launched (a chunk past the count exits at once)
    const int64_t rows_total = n_dec ? capacity : n_fixed;
    for (int64_t row0 = 0; row0 < rows_total; row0 += chunk_rows) {
        const int64_t rows = rows_total - row0 < chunk_rows ? rows_total - row0 : chunk_rows;
        const int64_t tiles_max = (rows + pol::TILE_M - 1) / pol::TILE_M;
        const int grid = (int)(tiles_max < h->sm_count ? tiles_max : h->sm_count);
        F.row0 = row0; F.rows_max = rows;
        upd::k_update_fwd_bwd<<<grid, pol::THREADS, pol::SMEM_BYTES, st>>>(F);
        CHECK_LAUNCH();
        D.row0 = row0; D.rows_max = rows;
        upd::k_update_dw<<<dw_grid, upd::DW_THREADS, dw_smem, st>>>(D);
        CHECK_LAUNCH();
    }
    return 0;
}

}  // extern "C"
