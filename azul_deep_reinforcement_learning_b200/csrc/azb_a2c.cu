// azb_a2c.cu -- the loss of Agent.update (reference azulnet/agent.py:45-56 with the per-decision terms of
// nn_runner.py:32-40) and its gradient with respect to the network outputs, for a batch of recorded decisions.
//
//   log_prob = log_softmax(masked logits)[action]            nn_runner.py:32, model.py:37-40
//   entropy  = -mean(log_softmax over the legal actions)     nn_runner.py:36-40 (the reference's "entropy")
//   advantage = q - value                                    agent.py:45 (NOT detached in the actor term)
//   loss = sum_n [ actor_c * (-log_prob * advantage) + critic_c * advantage^2 + entropy_c * entropy ] * scale
//
// One warp per decision: the 180 logits are read once (coalesced), max / sum-exp / legal-sum are warp
// reductions, the gradient row is written once.  HBM-bound: 2 x 720 B per decision.
#include <cuda_runtime.h>
#include <stdint.h>

#include "azb_internal.h"

namespace a2c {

constexpr int ACT = 180, PER_LANE = 6;      // columns lane, lane + 32, ...: 6 * 32 = 192 >= 180

__device__ __forceinline__ float warp_max(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xFFFFFFFFu, v, o));
    return v;
}
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}

struct Args {
    int64_t n;
    const float* __restrict__ logits;       // [n][180] raw (unmasked) actor outputs
    const float* __restrict__ value;        // [n]
    const uint32_t* __restrict__ mask_rows; // [n][6] legal-mask words of the decision (word p bit b <=> action 30p + b)
    const int64_t* __restrict__ action;     // [n]
    const float* __restrict__ qval;         // [n] discounted return
    float scale, actor_c, critic_c, entropy_c;
    float* __restrict__ dlogits;            // [n][180] d loss / d logits
    float* __restrict__ dvalue;             // [n]      d loss / d value
    double* __restrict__ sums;              // [3] += sum of (-log_prob * advantage), advantage^2, entropy (unscaled)
};

__global__ void __launch_bounds__(256) k_a2c_loss_grad(Args A)
{
    __shared__ double part[3][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
    double acc_a = 0.0, acc_c = 0.0, acc_e = 0.0;           // lane 0 accumulates this warp's rows
    for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp; row < A.n; row += warps_total) {
        const float* lr = A.logits + row * ACT;
        const uint32_t mw = lane < 6 ? A.mask_rows[row * 6 + lane] : 0u;
        float l[PER_LANE];
        bool legal[PER_LANE];
        const int act = (int)A.action[row];
        float mx = -INFINITY, sl = 0.0f;
        int k = 0;
        bool act_legal = false;
#pragma unroll
        for (int j = 0; j < PER_LANE; j++) {
            const int a = lane + 32 * j;
            const int p = a / 30, b = a - 30 * p;
            const uint32_t w = __shfl_sync(0xFFFFFFFFu, mw, p < 6 ? p : 0);
            legal[j] = a < ACT && ((w >> b) & 1u);
            l[j] = a < ACT ? lr[a] : 0.0f;
            if (legal[j]) { mx = fmaxf(mx, l[j]); sl += l[j]; k++; }
            act_legal |= legal[j] && a == act;
        }
        mx = warp_max(mx);
        float se = 0.0f;
#pragma unroll
        for (int j = 0; j < PER_LANE; j++) se += legal[j] ? expf(l[j] - mx) : 0.0f;
        se = warp_sum(se);
        sl = warp_sum(sl);
        k = (int)warp_sum((float)k);
        const float v = A.value[row], q = A.qval[row];
        float* dr = A.dlogits + row * ACT;
        // the lane holding the action reports whether it is legal: rows without a legal action or whose action is not
        // legal (model.py:33-34 IllegalMask: such rows are never recorded) contribute nothing
        if (!__any_sync(0xFFFFFFFFu, act_legal)) {
#pragma unroll
            for (int j = 0; j < PER_LANE; j++)
                if (lane + 32 * j < ACT) dr[lane + 32 * j] = 0.0f;
            if (lane == 0) A.dvalue[row] = 0.0f;
            continue;
        }
        const float lse = mx + logf(se);
        float la = 0.0f;                                    // logit of the taken action, from the lane that holds it
#pragma unroll
        for (int j = 0; j < PER_LANE; j++) la += (lane + 32 * j == act) ? l[j] : 0.0f;
        la = warp_sum(la);
        const float log_prob = la - lse;
        const float adv = q - v;
        const float inv_k = 1.0f / (float)k;
        const float entropy = -(sl * inv_k - lse);
#pragma unroll
        for (int j = 0; j < PER_LANE; j++) {
            const int a = lane + 32 * j;
            if (a < ACT) {
                float gj = 0.0f;
                if (legal[j]) {
                    const float pj = expf(l[j] - lse);
                    // d(-log_prob * adv)/dl_j = -adv * (delta_ja - p_j);  d entropy / dl_j = p_j - 1/k
                    gj = A.actor_c * (-adv) * ((a == act ? 1.0f : 0.0f) - pj) + A.entropy_c * (pj - inv_k);
                }
                dr[a] = gj * A.scale;
            }
        }
        if (lane == 0) {
            // value enters through advantage = q - value in the actor AND the critic term (agent.py:45-50)
            A.dvalue[row] = (A.actor_c * log_prob - 2.0f * A.critic_c * adv) * A.scale;
            acc_a += (double)(-log_prob * adv); acc_c += (double)(adv * adv); acc_e += (double)entropy;
        }
    }
    if (lane == 0) { part[0][warp] = acc_a; part[1][warp] = acc_c; part[2][warp] = acc_e; }
    __syncthreads();
    if (threadIdx.x < 3 && A.sums) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += part[threadIdx.x][w];
        atomicAdd(&A.sums[threadIdx.x], t);
    }
}

// Discounted returns of NNRunner.train (nn_runner.py:72-75) over the decision records of azb_policy_rollout's runner mode:
// one thread per game walks its decisions backwards, q = r + gamma * q (double, like the reference's numpy loop; the
// reference then casts to float32, agent.py:41), and scatters q to the decision's compact slot.
__global__ void k_returns(int64_t n, int k, double gamma, const int16_t* __restrict__ reward_rec,
                          const uint8_t* __restrict__ flags_rec, const int32_t* __restrict__ slot_rec,
                          float* __restrict__ qval, double* __restrict__ reward_sum, const uint32_t* __restrict__ steps_used)
{
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (steps_used && (int)*steps_used < k) k = (int)*steps_used;      // decision iterations the rollout actually ran
    // one running return per seat, picked by flags bit 2 (two-seat self-play records seat 2's decisions with it; the runner
    // modes never set it, so their returns are those of the one recurrence)
    double q1 = 0.0, q2 = 0.0, total = 0.0;
    if (g < n) {
        // backwards in groups of four: the twelve loads of a group are independent of the recurrence and in flight together
        for (int t1 = k; t1 > 0; t1 -= 4) {
            uint8_t f[4]; int16_t r[4]; int32_t sl[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int t = t1 - 1 - j;
                const int64_t i = (int64_t)(t < 0 ? 0 : t) * n + g;
                f[j] = t >= 0 ? flags_rec[i] : (uint8_t)0; r[j] = reward_rec[i]; sl[j] = slot_rec[i];
            }
#pragma unroll
            for (int j = 0; j < 4; j++) {
                if (!(f[j] & 1)) continue;
                const bool seat2 = (f[j] & 4) != 0;
                const double q = (double)r[j] + gamma * (seat2 ? q2 : q1);
                if (seat2) q2 = q; else q1 = q;
                total += (double)r[j];
                if (sl[j] >= 0) qval[sl[j]] = (float)q;
            }
        }
    }
    if (reward_sum) {                                   // sum of the episode rewards (Agent.update's "reward" statistic, agent.py:58)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xFFFFFFFFu, total, o);
        if ((threadIdx.x & 31) == 0 && total != 0.0) atomicAdd(reward_sum, total);
    }
}

// The statistics vector of one training batch in one pass over the games (what Agent.update / GameRunner's statistics
// report, agent.py:58-59, game_runner.py:10-22, azul.py:314-315): out[18] (double, zeroed by the caller) =
//   0 decision count (clamped to the record capacity), 1-3 the three loss sums, 4 sum of rewards, 5 games,
//   6-15 sums of Azul.get_statistics' ten raw values over the games, 16 games seat 1 won, 17 games not finished
//   (+ 1e9 when the decision records overflowed their capacity).
__global__ void k_train_stats(const uint32_t* __restrict__ s, int64_t n, const uint32_t* __restrict__ n_dec, int64_t rec_cap,
                              const double* __restrict__ loss_sums, const double* __restrict__ reward_sum, double* __restrict__ out)
{
    __shared__ double part[12][8];
    const int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double v[12];
#pragma unroll
    for (int i = 0; i < 12; i++) v[i] = 0.0;
    if (g < n) {                                                        // 2-player layout: MISC word 3, per player 7 + 5p .. 11 + 5p
        const uint32_t misc = s[3 * n + g], scf0 = s[9 * n + g], scf1 = s[14 * n + g], sta0 = s[10 * n + g], sta1 = s[15 * n + g], stb0 = s[11 * n + g];
        const double s0 = (double)(scf0 & 0xFFFFu), s1 = (double)(scf1 & 0xFFFFu);
        v[0] = s0; v[1] = s1; v[2] = (double)((misc >> 16) & 0xFFFu); v[3] = (double)(sta0 & 0xFFFu);
        v[4] = (double)((sta0 & 0xFFFu) + (sta1 & 0xFFFu)); v[5] = (double)((sta0 >> 12) & 0xFFFFu); v[6] = (double)(sta0 >> 28);
        v[7] = (double)(stb0 & 255u); v[8] = (double)((stb0 >> 16) & 255u); v[9] = (double)((stb0 >> 8) & 255u);
        v[10] = s0 > s1 ? 1.0 : 0.0; v[11] = ((misc >> 12) & 1u) ? 0.0 : 1.0;
    }
#pragma unroll
    for (int i = 0; i < 12; i++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_xor_sync(0xFFFFFFFFu, v[i], o);
        if ((threadIdx.x & 31) == 0) part[i][threadIdx.x >> 5] = v[i];
    }
    __syncthreads();
    if (threadIdx.x < 12) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += part[threadIdx.x][w];
        if (t != 0.0) atomicAdd(out + 6 + threadIdx.x, t);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const int64_t nd = (int64_t)*n_dec;
        out[0] = (double)(nd < rec_cap ? nd : rec_cap);
        out[1] = loss_sums[0]; out[2] = loss_sums[1]; out[3] = loss_sums[2];
        out[4] = reward_sum[0]; out[5] = (double)n;
        if (nd > rec_cap) atomicAdd(out + 17, 1e9);
    }
}

}  // namespace a2c

extern "C" int azb_train_stats(azb_t* h, const uint32_t* state, const uint32_t* n_dec, int64_t rec_cap, const double* loss_sums,
                               const double* reward_sum, double* out18, void* stream)
{
    CHECK_HANDLE(h);
    if (!state || !n_dec || !loss_sums || !reward_sum || !out18) return azb_fail(AZB_E_INVALID, "null buffer%s");
    if (h->players != 2) return azb_fail(AZB_E_INVALID, "training statistics are defined for the 2-player GameRunner%s");
    AZB_CUDA(cudaMemsetAsync(out18, 0, 18 * sizeof(double), (cudaStream_t)stream));
    a2c::k_train_stats<<<(unsigned)((h->n_games + 255) / 256), 256, 0, (cudaStream_t)stream>>>(state, h->n_games, n_dec, rec_cap,
                                                                                              loss_sums, reward_sum, out18);
    CHECK_LAUNCH();
    return 0;
}

extern "C" int azb_discounted_returns(azb_t* h, int k_decisions, double gamma, const int16_t* reward_rec,
                                      const uint8_t* flags_rec, const int32_t* slot_rec, float* qval, double* reward_sum,
                                      const uint32_t* steps_used, void* stream)
{
    CHECK_HANDLE(h);
    if (k_decisions < 0) return azb_fail(AZB_E_INVALID, "k_decisions < 0%s");
    if (!reward_rec || !flags_rec || !slot_rec || !qval) return azb_fail(AZB_E_INVALID, "null buffer%s");
    a2c::k_returns<<<(unsigned)((h->n_games + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        h->n_games, k_decisions, gamma, reward_rec, flags_rec, slot_rec, qval, reward_sum, steps_used);
    CHECK_LAUNCH();
    return 0;
}

extern "C" int azb_a2c_loss_grad(azb_t* h, int64_t n, const float* logits, const float* value, const uint32_t* mask_rows,
                                 const int64_t* action, const float* qval, float scale, float actor_coeff,
                                 float critic_coeff, float entropy_coeff, float* dlogits, float* dvalue, double* sums,
                                 void* stream)
{
    CHECK_HANDLE(h);
    if (n < 0) return azb_fail(AZB_E_INVALID, "n < 0%s");
    if (n == 0) return 0;
    if (!logits || !value || !mask_rows || !action || !qval || !dlogits || !dvalue) return azb_fail(AZB_E_INVALID, "null buffer%s");
    a2c::Args A{n, logits, value, mask_rows, action, qval, scale, actor_coeff, critic_coeff, entropy_coeff, dlogits, dvalue, sums};
    const int64_t blocks_needed = (n + 7) / 8;
    const int64_t cap = (int64_t)h->sm_count * 8;
    a2c::k_a2c_loss_grad<<<(unsigned)(blocks_needed < cap ? blocks_needed : cap), 256, 0, (cudaStream_t)stream>>>(A);
    CHECK_LAUNCH();
    return 0;
}
