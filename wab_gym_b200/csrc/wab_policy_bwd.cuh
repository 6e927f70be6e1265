// wab_policy_bwd.cuh — the vector-Jacobian product of the reference's Policy.forward (actor_critic.py:84-97) on the
// 5th-generation tensor cores: for T steps of N environments (rows t N + n) with upstream gradients g_logp, g_value of
// the sampled action's log-probability and of the value, the gradient of sum_rows g_logp log pi(a | x) + g_value V(x)
// with respect to all ten parameters of Policy. Included by wab_kernels.cu after wab_policy_tc.cuh.
//
// Training keeps only what the rollout produced (28 feature bytes, the action, the step's noise counter): a CTA owns a
// tile of 128 active rows and
//   1. recomputes the forward with the op sequence of wab_affine1_tc_kernel<2> (input generated in shared memory from the
//      feature bytes and the keyed noise, bf16 x 3 splits, the same accumulator split and epilogues), so the recomputed
//      log-probabilities and values equal the rollout's bit for bit;
//   2. d logits_i = g_logp (1[i = a] - p_i), d value = g_value; g3 = (W_heads^T d heads) * clamp mask * leaky'(z3);
//   3. dh2 = g3 W3 and dh1 = g2 W2 on the tensor cores, with W3^T and W2^T packed by wab_policy_linear_prepare into the
//      layouts of the forward's layer-2 and layer-3 loops (which this file runs again);
//   4. the weight gradients with K = the tile's 128 rows: both operands are written transposed from registers into the
//      canonical K-major layout (operand row = a feature, K = the tile's row), split three ways, six products per K step;
//      dW1 = g1^T x with x regenerated per 64-column slab and never written to memory;
//   5. reads each accumulator back after the tile (128 rows per tensor-memory accumulation) and adds it with
//      round-to-nearest fp32 adds into partial sums the CTA owns exclusively; bias gradients are butterfly sums.
// A persistent grid walks the tiles of the active rows (count read on the device); wab_policy_bwd_reduce_kernel then sums
// the per-CTA partials in a fixed order in fp64. No float atomics: equal inputs give bit-identical gradients.
// The hidden activations h1, h2 of the tile wait in a per-CTA stash in global memory (read back by the thread that wrote
// them) rather than in registers: the forward recompute already needs 128 registers a thread.
//
// wab_policy_ppo_bwd_kernel is the same pass with PPO's clipped objective in place of the upstream gradients (step 2):
// per row  l = -w_pi min(r A, clip(r, 1 - eps, 1 + eps) A) + w_v (V - R)^2 / 2 - w_H H,  r = exp(log pi(a | x) - logp_old),
// H = -sum_o p_o log p_o, with A, R, logp_old read per row. Its upstream gradients are closed forms of what the heads block
// already holds: g_logp = -w_pi A r (0 where the clip is active), g_value = w_v (V - R), and the entropy adds
// w_H p_o (log p_o + H) to d logit_o. Everything after the heads is shared.
//
// Two more kernels of the same body serve any loss written in torch over (logits, value). They take a LIST of M rows
// (ListArgs: a host count, B.rows or NULL for row m = m) and index their inputs and outputs by the list position m, so a
// minibatch needs no [T, N] arrays; a listed entry outside [0, T N) gets NaN outputs and contributes nothing:
//   wab_policy_eval_kernel        step 1 and the heads only: logits [M][A] (before the softmax, bias included), value [M];
//   wab_policy_logits_bwd_kernel  the whole pass with d heads read per row (d logits [M][A], d value [M]) in step 2.
#pragma once

namespace {

constexpr uint32_t BW_LEAD = 256;                   // tensor-memory columns of the leading-product accumulators (of 512)
constexpr int BW_KROW = 2048;                       // bytes between 8-operand-row groups of a K = 128 operand
constexpr int BW_M_PART = 128 * 256;                // one bf16 part of a 128-row, K = 128 operand: 32 KB
constexpr int BW_SMEM_M = 0, BW_SMEM_N = 3 * BW_M_PART, BW_SMEM_BITS = BW_SMEM_N + 3 * 80 * 256,
              BW_SMEM_WSM = BW_SMEM_BITS + TC_TILE_M * TC_ROWBITS_STRIDE * 4, BW_SMEM_PART = BW_SMEM_WSM + 12 * 128 * 4,
              BW_SMEM_DH = BW_SMEM_PART + 128 * 2 * 9 * 4, BW_SMEM_RED = BW_SMEM_DH + 128 * 9 * 4,
              BW_SMEM_BAR = BW_SMEM_RED + 4 * 160 * 4, BW_SMEM_TOTAL = BW_SMEM_BAR + 16;
// per-CTA partial sums (floats): dW1 [slab c][out j][slab column 64], b1, dW2^T [in 128][out 160], b2, dW3 [out 128][in 160],
// b3, dW_heads^T [in 128][16], b_heads [16]; then the stash h1 [128][128], h2 [128][160]
constexpr int BP_W1 = 0, BP_B1 = BP_W1 + 8 * 128 * 64, BP_W2T = BP_B1 + 128, BP_B2 = BP_W2T + 128 * 160, BP_W3 = BP_B2 + 160,
              BP_B3 = BP_W3 + 128 * 160, BP_WH = BP_B3 + 128, BP_BH = BP_WH + 128 * 16, BP_PARTIAL = BP_BH + 16,
              BP_H1 = BP_PARTIAL, BP_H2 = BP_H1 + 128 * 128, BP_BLOCK = BP_H2 + 128 * 160;

struct BackwardArgs {
    const uint8_t* features;                 // u8[T][N][28]
    int64_t n_envs, n_rows;                  // N, T N
    const unsigned long long* counters;      // the noise counter of each step, [T]
    const uint8_t* actions; const float* g_logp; const float* g_value;
    const int32_t* rows; const long long* d_count;    // active rows and their count (both NULL: every row)
    const uint4* w1; const float* b1; const uint4* w2; const float* b2; const uint4* w3; const float* b3;
    const uint4* w2t; const uint4* w3t;      // W2^T [128][150], W3^T [150][128] packed by wab_policy_linear_prepare
    const float* w_heads; const float* b_heads;
    int n_actions; float noise_scale, slope, clamp_lo, clamp_hi;
    float* scratch;                          // gridDim.x blocks of BP_BLOCK floats
    float* logp_out; float* value_out;       // recomputed log pi(a | x), V(x) per row (optional)
};

// the PPO objective of wab_policy_ppo_bwd_kernel (g_logp / g_value of BackwardArgs are unused there)
struct PpoArgs {
    const float* logp_old; const float* advantage; const float* target;   // per row
    float clip_eps, w_policy, w_value, w_entropy;
    float* entropy_out;                      // H per row (optional)
};

// the list kernels (wab_policy_eval_kernel, wab_policy_logits_bwd_kernel): M = n_list rows, row m = B.rows[m] (B.rows
// NULL: m); arrays indexed by m. B.d_count, B.actions, B.g_logp, B.g_value, B.logp_out and B.value_out are unused there
struct ListArgs {
    long long n_list;                        // M (a host count; may exceed T N when rows repeat)
    const float* g_logits; const float* g_value;       // upstream d logits [M][A], d value [M] (the logits backward)
    float* logits_out; float* value_out;     // logits [M][A], value [M] (the evaluation)
};

// which heads block the body runs (step 2), and whether steps 3 - 5 follow (not for BW_EVAL); BW_PPO_POP is BW_PPO for
// one member of a population (wab_policy_ppo_bwd_population_kernel)
enum BwKind { BW_A2C, BW_PPO, BW_EVAL, BW_LOGITS, BW_PPO_POP };

// the CTA's member in wab_policy_ppo_bwd_population_kernel; the other kernels declare an unused one
struct MemberArgs {
    int member, cta, n_cta;                  // member m = blockIdx.x / n_cta, its local CTA index cta = blockIdx.x % n_cta
    long long member_envs, list_len;         // n: member m owns envs [m n, (m + 1) n); M: entries of its row list
};

// element (operand row n, K = tile row k) of a K = 128 operand, canonical K-major layout without swizzle
__device__ __forceinline__ uint32_t bw_off(int n, int k) { return (uint32_t)((n >> 3) * BW_KROW + (k >> 3) * 128 + (n & 7) * 16 + (k & 7) * 2); }
__device__ __forceinline__ void bw_st16(uint32_t addr, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" :: "r"(addr), "h"((unsigned short)v) : "memory"); }
// v split three ways into the parts of an operand (part stride `part` bytes) at element (n, k)
__device__ __forceinline__ void bw_put(uint32_t base, uint32_t part, int n, int k, float v) {
    uint32_t p0, p1, p2;
    tc_split3(v, p0, p1, p2);
    const uint32_t a = base + bw_off(n, k);
    bw_st16(a, p0); bw_st16(a + part, p1); bw_st16(a + 2 * part, p2);
}
// sum over the 32 rows of a warp (butterfly: the same order every time)
__device__ __forceinline__ float bw_warp_sum(float v) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, s);
    return v;
}

// column sums of a [128 rows][2 halves x CNT] matrix held a row-half per thread (thread = row tid & 127, half tid >> 7):
// warp butterflies, then the four warps of a half in index order; adds into dst[j] for j < valid
template <int CNT>
__device__ __forceinline__ void bw_bias_sum(const float (&g)[CNT], int valid, float* red, float* dst) {
    const int tid = threadIdx.x, q = (tid >> 5) & 3, h = tid >> 7;
#pragma unroll
    for (int j = 0; j < CNT; ++j) {
        const float s = bw_warp_sum(g[j]);
        if ((tid & 31) == 0) red[q * 160 + h * CNT + j] = s;
    }
    __syncthreads();
    for (int j = tid; j < valid; j += 256) dst[j] += ((red[j] + red[160 + j]) + red[320 + j]) + red[480 + j];
    __syncthreads();
}

__global__ void __launch_bounds__(256, 1)
wab_policy_bwd_kernel(const __grid_constant__ Params P, int food_dim, const __grid_constant__ BackwardArgs B) {
    constexpr BwKind KIND = BW_A2C;
    const PpoArgs Q{};
    const ListArgs L{};
    const MemberArgs G{};
#include "wab_policy_bwd_body.cuh"
}

__global__ void __launch_bounds__(256, 1)
wab_policy_ppo_bwd_kernel(const __grid_constant__ Params P, int food_dim, const __grid_constant__ BackwardArgs B,
                          const __grid_constant__ PpoArgs Q) {
    constexpr BwKind KIND = BW_PPO;
    const ListArgs L{};
    const MemberArgs G{};
#include "wab_policy_bwd_body.cuh"
}

#pragma nv_diag_suppress 128                        // steps 3 - 5 of the body, after the evaluation's `continue`
__global__ void __launch_bounds__(256, 1)
wab_policy_eval_kernel(const __grid_constant__ Params P, int food_dim, const __grid_constant__ BackwardArgs B,
                       const __grid_constant__ ListArgs L) {
    constexpr BwKind KIND = BW_EVAL;
    const PpoArgs Q{};
    const MemberArgs G{};
#include "wab_policy_bwd_body.cuh"
}
#pragma nv_diag_default 128

__global__ void __launch_bounds__(256, 1)
wab_policy_logits_bwd_kernel(const __grid_constant__ Params P, int food_dim, const __grid_constant__ BackwardArgs B,
                             const __grid_constant__ ListArgs L) {
    constexpr BwKind KIND = BW_LOGITS;
    const PpoArgs Q{};
    const MemberArgs G{};
#include "wab_policy_bwd_body.cuh"
}

// the population backward: P members of n envs each on ONE grid of P n_cta CTAs (n_cta = the single-policy grid). CTA b
// serves member m = b / n_cta as local CTA c = b % n_cta and walks tiles c, c + n_cta, ... of m's row list: the tiles a
// single-policy launch gives its CTA c, into the scratch block b = m n_cta + c, so member m's partial sums are those of
// its own wab_policy_ppo_bwd_kernel bit for bit. Weights are stacked per member at the packers' strides.
struct PopulationArgs {
    int n_cta;
    long long member_envs, list_len;         // n, M
    const int32_t* rows; const long long* counts;    // [P][M] global rows t N + n, [P] counts (read on the device)
    float coef[64][4];                       // clip_eps, w_policy, w_value, w_entropy of each member
};

__global__ void __launch_bounds__(256, 1)
wab_policy_ppo_bwd_population_kernel(const __grid_constant__ Params P, int food_dim, const __grid_constant__ BackwardArgs Bs,
                                     const __grid_constant__ PpoArgs Qs, const __grid_constant__ PopulationArgs Pop) {
    constexpr BwKind KIND = BW_PPO_POP;
    const ListArgs L{};
    const int m = (int)(blockIdx.x / (unsigned)Pop.n_cta);
    const MemberArgs G{m, (int)blockIdx.x - m * Pop.n_cta, Pop.n_cta, Pop.member_envs, Pop.list_len};
    const int64_t heads_n = Bs.n_actions + 1;
    BackwardArgs B = Bs;
    B.rows = Pop.rows + m * Pop.list_len; B.d_count = Pop.counts + m;
    B.w1 += m * POP_W1_U4; B.b1 += m * 128; B.w2 += m * POP_LINEAR_U4; B.b2 += m * 150; B.w3 += m * POP_LINEAR_U4;
    B.b3 += m * 128; B.w2t += m * POP_LINEAR_U4; B.w3t += m * POP_LINEAR_U4; B.w_heads += m * heads_n * 128; B.b_heads += m * heads_n;
    PpoArgs Q = Qs;
    Q.clip_eps = Pop.coef[m][0]; Q.w_policy = Pop.coef[m][1]; Q.w_value = Pop.coef[m][2]; Q.w_entropy = Pop.coef[m][3];
#include "wab_policy_bwd_body.cuh"
}

// the per-CTA partial sums -> the flat gradient in parameters_to_vector(Policy.parameters()) order, summed over the CTAs
// in index order in fp64. G = float rounds once (wab_policy_backward); G = double keeps the fp64 sum
// (wab_policy_backward_grad_f64, for a cross-rank sum that rounds once at its end)
template <typename G>
__global__ void wab_policy_bwd_reduce_kernel(const float* __restrict__ scratch, int n_blocks, int dim, int n_actions, G* __restrict__ grad) {
    const int64_t n1 = 128LL * dim, o_b1 = n1, o_w2 = o_b1 + 128, o_b2 = o_w2 + 150 * 128, o_w3 = o_b2 + 150, o_b3 = o_w3 + 128 * 150,
                  o_wa = o_b3 + 128, o_ba = o_wa + (int64_t)n_actions * 128, o_wv = o_ba + n_actions, o_bv = o_wv + 128, total = o_bv + 1;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    int off;
    if (e < o_b1) {
        const int j = (int)(e / dim), k = (int)(e - (int64_t)j * dim);
        const int c = 2 * (k >> 7) + ((k >> 4) & 1), s = (k >> 5) & 3, hh = (k >> 3) & 1, el = k & 7;   // tc_column inverted
        off = BP_W1 + (c * 128 + j) * 64 + 8 * (4 * hh + s) + el;
    } else if (e < o_w2) off = BP_B1 + (int)(e - o_b1);
    else if (e < o_b2) { const int j = (int)((e - o_w2) / 128), i = (int)((e - o_w2) % 128); off = BP_W2T + i * 160 + j; }
    else if (e < o_w3) off = BP_B2 + (int)(e - o_b2);
    else if (e < o_b3) { const int j = (int)((e - o_w3) / 150), i = (int)((e - o_w3) % 150); off = BP_W3 + j * 160 + i; }
    else if (e < o_wa) off = BP_B3 + (int)(e - o_b3);
    else if (e < o_ba) { const int o = (int)((e - o_wa) / 128), i = (int)((e - o_wa) % 128); off = BP_WH + i * 16 + o; }
    else if (e < o_wv) off = BP_BH + (int)(e - o_ba);
    else if (e < o_bv) off = BP_WH + (int)(e - o_wv) * 16 + n_actions;
    else off = BP_BH + n_actions;
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += (double)scratch[(size_t)b * BP_BLOCK + off];
    grad[e] = (G)s;
}

// wab_policy_bwd_reduce_kernel for each member of a population (blockIdx.y = m): the fp64 sum over m's own n_cta CTAs, in
// index order, into grad [P][stride]. G = float rounds once (wab_policy_ppo_backward_population); G = double keeps the
// fp64 sum (wab_policy_backward_population_grad_f64, for a cross-rank sum) and, launched over the whole stride, also
// writes the padding entries as 0. The element -> partial-sum mapping is restated rather than shared: moved into a
// device function, it compiles differently inside wab_policy_bwd_reduce_kernel.
template <typename G>
__global__ void wab_policy_bwd_reduce_population_kernel(const float* __restrict__ scratch, int n_cta, int dim, int n_actions,
                                                        int64_t stride, G* __restrict__ grad) {
    const int64_t n1 = 128LL * dim, o_b1 = n1, o_w2 = o_b1 + 128, o_b2 = o_w2 + 150 * 128, o_w3 = o_b2 + 150, o_b3 = o_w3 + 128 * 150,
                  o_wa = o_b3 + 128, o_ba = o_wa + (int64_t)n_actions * 128, o_wv = o_ba + n_actions, o_bv = o_wv + 128, total = o_bv + 1;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) {
        if (sizeof(G) == 8 && e < stride) grad[(int64_t)blockIdx.y * stride + e] = (G)0;
        return;
    }
    int off;
    if (e < o_b1) {
        const int j = (int)(e / dim), k = (int)(e - (int64_t)j * dim);
        const int c = 2 * (k >> 7) + ((k >> 4) & 1), s = (k >> 5) & 3, hh = (k >> 3) & 1, el = k & 7;   // tc_column inverted
        off = BP_W1 + (c * 128 + j) * 64 + 8 * (4 * hh + s) + el;
    } else if (e < o_w2) off = BP_B1 + (int)(e - o_b1);
    else if (e < o_b2) { const int j = (int)((e - o_w2) / 128), i = (int)((e - o_w2) % 128); off = BP_W2T + i * 160 + j; }
    else if (e < o_w3) off = BP_B2 + (int)(e - o_b2);
    else if (e < o_b3) { const int j = (int)((e - o_w3) / 150), i = (int)((e - o_w3) % 150); off = BP_W3 + j * 160 + i; }
    else if (e < o_wa) off = BP_B3 + (int)(e - o_b3);
    else if (e < o_ba) { const int o = (int)((e - o_wa) / 128), i = (int)((e - o_wa) % 128); off = BP_WH + i * 16 + o; }
    else if (e < o_wv) off = BP_BH + (int)(e - o_ba);
    else if (e < o_bv) off = BP_WH + (int)(e - o_wv) * 16 + n_actions;
    else off = BP_BH + n_actions;
    const float* member = scratch + (size_t)blockIdx.y * n_cta * BP_BLOCK;
    double s = 0.0;
    for (int b = 0; b < n_cta; ++b) s += (double)member[(size_t)b * BP_BLOCK + off];
    grad[(int64_t)blockIdx.y * stride + e] = (G)s;
}

// d_grad[i] = fp32(sum over r = 0 .. n_ranks - 1 of d_rank_grads[r][i]), the sum in fp64 in rank order
__global__ void wab_policy_grad_sum_ranks_kernel(const double* __restrict__ rank_grads, int n_ranks, int64_t n, float* __restrict__ grad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s = 0.0;
    for (int r = 0; r < n_ranks; ++r) s += rank_grads[(size_t)r * n + i];
    grad[i] = (float)s;
}

}  // namespace
