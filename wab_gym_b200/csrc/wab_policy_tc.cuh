// wab_policy_tc.cuh — the first layer of the reference's Policy (actor_critic.py:59, :88-90) on the 5th-generation tensor
// cores: h1 = leaky_relu(affine1(flatten(obs) + U[0,1)/100)) for a batch of environments, straight from the 28 feature
// bytes per environment (wab_features.cuh). Included by wab_kernels.cu.
//
// This is the one dense contraction on the consumer side of the path (32,768 x 449 x 128 per rollout step). The library
// route is three passes — write the 449-wide input (wab_flatten_noisy_kernel), an fp32 SIMT GEMM (cuBLAS), the activation —
// and spends 54 us of a 281 us rollout step in the GEMM alone. Here ONE kernel does all of it and the input matrix never
// exists in HBM:
//   * a CTA owns a tile of 128 environments; its 256 threads GENERATE the A operand of each K-chunk in shared memory:
//     the one-hot columns from the feature bytes, the same keyed noise as wab_flatten_noisy_kernel (one Philox4x32 call
//     per 4 columns), x = onehot + scale * u in fp32 exactly as that kernel computes it;
//   * fp32 accuracy on bf16 tensor cores: W is split into three bf16 terms (W = W0 + W1 + W2, 24 mantissa bits) and x into
//     its one-hot part o (0 or 1: exact in bf16) and its noise part n = x - o (exact in fp32; n = n0 + n1 to 2^-16 of
//     its size, which is <= noise_scale); six products are accumulated in fp32 in tensor memory:
//     o W0 + o W1 + o W2 + n0 W0 + n0 W1 + n1 W0 (what is dropped is below 2^-24 of the sum, i.e. fp32 rounding);
//   * tcgen05.mma (M 128, N 128, K 16, kind::f16, operands by shared-memory descriptor, no swizzle), issued by one
//     thread, completion through tcgen05.commit on an mbarrier; accumulators read back with tcgen05.ld for the
//     epilogue (bias, leaky-ReLU, 16-byte stores of the 128 outputs).
//   * The K order inside the product is free, so it is chosen for the generator: chunk c (64 columns) holds the columns
//     k = 128 (c >> 1) + 32 s + j, s = 0..3, j = 16 (c & 1) .. + 16 — the four words of 16 Philox calls — and
//     wab_policy_affine1_prepare lays the split weights out in the same order (and in the canonical core-matrix
//     layout), once per weight update.
#pragma once

namespace {

constexpr int TC_TILE_M = 128;          // environments per CTA
constexpr int TC_N = 128;               // affine1 outputs (actor_critic.py:59)
constexpr int TC_KC = 64;               // K columns per chunk
constexpr int TC_CHUNKS = 8;            // 512 >= 449 columns (the padding columns are zero on both sides)
constexpr int TC_PART_BYTES = TC_TILE_M * TC_KC * 2;        // one bf16 operand part of one chunk: 16 KB
constexpr int TC_ROWBITS_STRIDE = 17;   // words per row of the one-hot bit vectors (16 + 1: conflict-free for a thread per row)
constexpr int TC_SMEM_A = 0, TC_SMEM_B = 3 * TC_PART_BYTES, TC_SMEM_BITS = 6 * TC_PART_BYTES,
              TC_SMEM_BAR = TC_SMEM_BITS + TC_TILE_M * TC_ROWBITS_STRIDE * 4, TC_SMEM_TOTAL = TC_SMEM_BAR + 16;

// canonical K-major layout without swizzle (UMMA "interleave"): core matrix = 8 rows x 16 bytes, contiguous (128 B);
// core matrices adjacent in K 128 B apart (leading byte offset), 8-row groups 1024 B apart (stride byte offset)
__host__ __device__ inline int tc_elem_offset(int row, int kc, int e) { return (row >> 3) * 512 + kc * 64 + (row & 7) * 8 + e; }
// chunk c, core-matrix column kc (0..7), element e (0..7) -> column of the 449-wide input (may be >= dim: padding)
__host__ __device__ inline int tc_column(int c, int kc, int e) {
    const int h = kc >> 2, s = kc & 3, j = 16 * (c & 1) + 8 * h + e;
    return 128 * (c >> 1) + 32 * s + j;
}

// matrix descriptor: start address, LBO 128 B (core matrices adjacent in K), SBO = 8-row group stride (16 bytes x the chunk's K), version 1, no swizzle
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t saddr, uint32_t sbo_bytes = 1024u) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// instruction descriptor, kind::f16: D fp32 (bits 4-5 = 1), A and B bf16 (bits 7-9, 10-12 = 1), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr uint32_t tc_idesc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TC_TILE_M >> 4) << 24);
}
constexpr uint32_t TC_IDESC = tc_idesc(TC_N);
constexpr int T2_KC = 32;                                  // layers 2 and 3: K columns per chunk
constexpr int T2_A_PART = TC_TILE_M * T2_KC * 2;           // 8 KB: one part of a 128-row operand chunk
constexpr int T2_B160_PART = 160 * T2_KC * 2;              // 10 KB: one part of a 160-row weight chunk

// 16-byte asynchronous global -> shared copy (LDGSTS) and the wait for all of this thread's copies
__device__ __forceinline__ void tc_cp_async16(uint32_t s_dst, const void* g_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(s_dst), "l"(g_src) : "memory");
}
__device__ __forceinline__ void tc_cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    unsigned long long t0 = 0ull;
    for (uint32_t spins = 0; !ok; ++spins) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (!ok && (spins & 1023u) == 1023u) {     // a wrong descriptor or phase must fail loudly within a second, never hang the device
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0ull) t0 = now;
            else if (now - t0 > 1000000000ull) __trap();
        }
    }
}
// v = p0 + p1 + p2 exactly (three bf16 terms carry 24 mantissa bits)
__device__ __forceinline__ void tc_split3(float v, uint32_t& p0, uint32_t& p1, uint32_t& p2) {
    const __nv_bfloat16 b0 = __float2bfloat16_rn(v);
    const float r1 = v - __bfloat162float(b0);
    const __nv_bfloat16 b1 = __float2bfloat16_rn(r1);
    const float r2 = r1 - __bfloat162float(b1);
    const __nv_bfloat16 b2 = __float2bfloat16_rn(r2);
    p0 = (uint32_t)__bfloat16_as_ushort(b0); p1 = (uint32_t)__bfloat16_as_ushort(b1); p2 = (uint32_t)__bfloat16_as_ushort(b2);
}

// W f32[128][dim] (nn.Linear weight) -> packed bf16 [chunk][part][tc_elem_offset(n, kc, e)], parts W0, W1, W2
__global__ void wab_affine1_prepare_kernel(const float* __restrict__ w, int dim, uint16_t* __restrict__ packed) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;            // (chunk, n, kc, e)
    if (idx >= TC_CHUNKS * TC_N * TC_KC) return;
    const int e = idx & 7, kc = (idx >> 3) & 7, n = (idx >> 6) & 127, c = idx >> 13;
    const int k = tc_column(c, kc, e);
    const float v = k < dim ? w[(int64_t)n * dim + k] : 0.f;
    uint32_t p0, p1, p2;
    tc_split3(v, p0, p1, p2);
    const int off = tc_elem_offset(n, kc, e), part = TC_TILE_M * TC_KC;
    packed[(c * 3 + 0) * part + off] = (uint16_t)p0;
    packed[(c * 3 + 1) * part + off] = (uint16_t)p1;
    packed[(c * 3 + 2) * part + off] = (uint16_t)p2;
}

// 32 consecutive accumulator columns of this thread's tensor-memory lane (issue only; tcgen05.wait::ld before use)
__device__ __forceinline__ void tc_tmem_ld32(uint32_t taddr, uint32_t v[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr) : "memory");
}

__device__ __forceinline__ void tc_tmem_ld16(uint32_t taddr, uint32_t v[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}

// W f32[n_out][n_in] (nn.Linear weight) -> bf16 [K chunk of 32][part][(n >> 3) * 256 + kcol * 64 + (n & 7) * 8 + e], n padded to
// n_pad rows and K to k_pad columns with zeros: the operand chunks of layers 2 and 3
__global__ void wab_linear_prepare_kernel(const float* __restrict__ w, int n_out, int n_in, int n_pad, int k_pad, uint16_t* __restrict__ packed) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;            // (n, k)
    if (idx >= n_pad * k_pad) return;
    const int n = idx / k_pad, k = idx - n * k_pad;
    const float v = (n < n_out && k < n_in) ? w[(int64_t)n * n_in + k] : 0.f;
    uint32_t p0, p1, p2;
    tc_split3(v, p0, p1, p2);
    const int chunk = k / T2_KC, kk = k - chunk * T2_KC, part = n_pad * T2_KC;
    const int off = (n >> 3) * (T2_KC * 8) + (kk >> 3) * 64 + (n & 7) * 8 + (kk & 7);
    packed[(chunk * 3 + 0) * part + off] = (uint16_t)p0;
    packed[(chunk * 3 + 1) * part + off] = (uint16_t)p1;
    packed[(chunk * 3 + 2) * part + off] = (uint16_t)p2;
}

// two fp32 -> one word of two bf16 (round to nearest even), `lo` in the low half
__device__ __forceinline__ uint32_t tc_pack_bf16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// TRUNK = false: out = h1 f32[rows][128] = leaky_relu(affine1(x)). TRUNK = true: the whole trunk of Policy.forward
// (actor_critic.py:88-92) without leaving the SM — h1 and h2 go from the accumulators through registers (bias, leaky-ReLU,
// three-way bf16 split) straight back into shared memory as the next layer's A operand — and out = z3 f32[rows][128], the
// PRE-activation output of affine3 (what wab_policy_tail takes).
struct TrunkWeights {
    const uint4* w2; const float* b2;      // affine2 128 -> 150, packed by wab_policy_linear_prepare (N padded to 160)
    const uint4* w3; const float* b3;      // affine3 150 -> 128 (K padded to 160)
    int n2;                                // 150
    // MODE 2 only — the tail of Policy.forward + select_action (actor_critic.py:92-97, :108-125), as wab_policy_tail_kernel
    uint32_t rk0[10], rk1[10];             // Philox round keys of the sampling seed
    const float* w_heads; const float* b_heads;   // f32[A + 1][128], f32[A + 1]: action_head stacked on value_head
    int n_actions; float clamp_lo, clamp_hi;
    uint8_t* actions; float* value; float* probs; float* logp;
    // MODES 4 and 5 only — a population of policies (wab_policy_forward_population, wab_policy_act_population): rows
    // [m member_rows, (m + 1) member_rows) take member m's weights, stacked per member at the strides below; member_rows is
    // a multiple of TC_TILE_M
    int64_t member_rows;
};
// per-member strides of the stacked packed weights, in uint4: wab_policy_affine1_packed_bytes() / 16 and
// wab_policy_linear_packed_bytes(n_out, n_in) / 16 of every layer of the reference's trunk (128 -> 150, 150 -> 128 and the
// transposes: 160 x 128 or 128 x 160 padded, three bf16 parts)
constexpr int64_t POP_W1_U4 = (int64_t)TC_CHUNKS * 3 * TC_PART_BYTES / 16, POP_LINEAR_U4 = 3 * 160 * 128 * 2 / 16;
// MODE 0: first layer only; 1: the trunk (out = z3); 2: trunk + tail (clamp, both heads, softmax, Categorical sample; out = z3 or null);
// 3: MODE 2 with the greedy action (the first index of the largest logit) instead of the sample: no Philox call, the round keys unread;
// 4: MODE 2 for a population: the CTA's rows are member row0 / member_rows's, and every weight pointer moves to that member's;
// 5: MODE 4 with MODE 3's greedy action
template <int MODE>
__global__ void __launch_bounds__(256, 2)
wab_affine1_tc_kernel(const __grid_constant__ Params P, const uint8_t* __restrict__ features, int64_t rows, int food_dim,
                      const uint4* __restrict__ wpacked, const float* __restrict__ bias, float noise_scale, float slope,
                      const unsigned long long* __restrict__ d_counter, float* __restrict__ out, TrunkWeights tw) {
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(tc_smem);
    const uint32_t s_a = s_base + TC_SMEM_A, s_b = s_base + TC_SMEM_B, s_bar = s_base + TC_SMEM_BAR;
    uint32_t* rowbits = reinterpret_cast<uint32_t*>(tc_smem + TC_SMEM_BITS);
    const int64_t row0 = (int64_t)blockIdx.x * TC_TILE_M;
    if constexpr (MODE == 4 || MODE == 5) {               // a CTA never straddles two members: member_rows % TC_TILE_M == 0
        const int64_t m = row0 / tw.member_rows, n_out = tw.n_actions + 1;
        wpacked += m * POP_W1_U4; bias += m * TC_N;
        tw.w2 += m * POP_LINEAR_U4; tw.b2 += m * tw.n2; tw.w3 += m * POP_LINEAR_U4; tw.b3 += m * TC_N;
        tw.w_heads += m * n_out * 128; tw.b_heads += m * n_out;
    }

    if (warp == 0) {                                      // two fp32 accumulators of 128 columns in tensor memory
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"((uint32_t)__cvta_generic_to_shared(&tmem_slot)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(s_bar), "r"(1u) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // ---- the one-hot part of the tile's rows as bit vectors (bit k = column k of gym.spaces.flatten, wab_env.py:710-724):
    // one thread per row walks the 28 features instead of the 449 columns
    if (tid >= 128) {
        const int rr = tid - 128;
        const int64_t grow = row0 + rr;
        uint32_t* bits = rowbits + rr * TC_ROWBITS_STRIDE;
#pragma unroll
        for (int k = 0; k < 16; ++k) bits[k] = 0u;
        if (grow < rows) {
            uint32_t fw[7];
#pragma unroll
            for (int k = 0; k < 7; ++k) fw[k] = reinterpret_cast<const uint32_t*>(features)[grow * 7 + k];
            auto fbyte = [&](int i) { return (int)((fw[i >> 2] >> (8 * (i & 3))) & 0xFFu); };
            auto hot = [&](int col) { bits[col >> 5] |= 1u << (col & 31); };
#pragma unroll
            for (int species = 0; species < 2; ++species) {
#pragma unroll
                for (int i = 0; i < 8; ++i) { const int v = fbyte(species * 12 + i); if (v < 12) hot(species * 140 + i * 12 + v); }
#pragma unroll
                for (int i = 0; i < 4; ++i) { const int v = fbyte(species * 12 + 8 + i); if (v < 11) hot(species * 140 + 96 + i * 11 + v); }
            }
            { const int v = fbyte(24); if (v < 2) hot(280 + v); }
            { const int v = fbyte(25); if (v < food_dim) hot(282 + v); }
            { const int v = fbyte(26); if (v < 2) hot(282 + food_dim + v); }
            { const int v = fbyte(27); if (v < 3) hot(284 + food_dim + v); }
            if (P.restrict_view) {                                    // the 121-cell view mask of the role (obs[6])
                const uint32_t* vm = fbyte(26) == 1 ? P.mask_gath : P.mask_look;
                const int base = 287 + food_dim;
#pragma unroll
                for (int wd = 0; wd < 4; ++wd) {
                    const uint32_t m = wd == 3 ? vm[3] & ((1u << (CELLS - 96)) - 1u) : vm[wd];
                    const int pos = base + 32 * wd;
                    bits[pos >> 5] |= m << (pos & 31);
                    if (pos & 31) bits[(pos >> 5) + 1] |= m >> (32 - (pos & 31));
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;

    const int r = tid & 127, h = tid >> 7;                // this thread's row of the tile and half of each chunk's lanes
    const int64_t row = row0 + r;
    const uint32_t* mybits = rowbits + r * TC_ROWBITS_STRIDE;
    const unsigned long long ctr = d_counter ? *d_counter : 0ull;
    const bool noisy = noise_scale != 0.f;
    const float scale = noise_scale * (1.0f / 16777216.0f);
    const uint32_t a_row = (uint32_t)((r >> 3) * 1024 + (r & 7) * 16);
    uint32_t parity = 0;

    for (int c = 0; c < TC_CHUNKS; ++c) {
        // ---- A: 8 Philox calls -> 32 columns of this row (4 core-matrix columns of 8): x = onehot + scale * m in fp32 exactly
        // as wab_flatten_noisy_kernel computes it; parts o (one-hot), n0, n1 (the noise x - o in two bf16 terms)
        float x[4][8];
        const int jb = 16 * (c & 1) + 8 * h;              // this thread's lanes j = jb .. jb + 7 of the chunk's Philox calls
        const uint64_t g = global_env_id(P, row);         // the noise key: the row's global env id
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            if (noisy)
                philox(P, (uint32_t)g, (uint32_t)(g >> 32) ^ ((uint32_t)(c >> 1) << 24) ^ ((uint32_t)(jb + e) << 16), (uint32_t)ctr,
                       (uint32_t)(ctr >> 32) ^ 0x464C4154u, w);
#pragma unroll
            for (int s = 0; s < 4; ++s) x[s][e] = scale * (float)(w[s] >> 8);
        }
        // The MMAs of the previous chunk (issued before this chunk's Philox calls started) have read both operand buffers by
        // now: start the asynchronous copy of this chunk's weights — 48 KB already in operand layout, 12 copies of 16 bytes per
        // thread, all in flight at once — and build the A operand's bf16 parts while it runs.
        if (c > 0) { tc_mbar_wait(s_bar, parity); parity ^= 1u; }
        {
            const uint4* src = wpacked + (size_t)c * (3 * TC_PART_BYTES / 16);
#pragma unroll
            for (int k = tid; k < 3 * TC_PART_BYTES / 16; k += 256) tc_cp_async16(s_b + (uint32_t)k * 16u, src + k);
        }
        uint32_t pk[3][4][4];                             // [part][s][word of the 16-byte vector]
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const uint32_t ob = (mybits[4 * (c >> 1) + s] >> jb) & 0xFFu;     // one-hot bits of columns 128 (c >> 1) + 32 s + jb ..
#pragma unroll
            for (int e2 = 0; e2 < 4; ++e2) {
                const float oa = (float)((ob >> (2 * e2)) & 1u), obb = (float)((ob >> (2 * e2 + 1)) & 1u);
                const float na = (oa + x[s][2 * e2]) - oa, nb = (obb + x[s][2 * e2 + 1]) - obb;   // the noise as it survives in x
                const uint32_t n0 = tc_pack_bf16x2(na, nb);
                const float ra = na - __uint_as_float(n0 << 16), rb = nb - __uint_as_float(n0 & 0xFFFF0000u);
                pk[0][s][e2] = (((ob >> (2 * e2)) & 1u) * 0x3F80u) | (((ob >> (2 * e2 + 1)) & 1u) * 0x3F800000u);
                pk[1][s][e2] = n0;
                pk[2][s][e2] = tc_pack_bf16x2(ra, rb);
            }
        }
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int s = 0; s < 4; ++s)
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(s_a + p * TC_PART_BYTES + a_row + (uint32_t)(h * 4 + s) * 128u),
                             "r"(pk[p][s][0]), "r"(pk[p][s][1]), "r"(pk[p][s][2]), "r"(pk[p][s][3]) : "memory");
        tc_cp_async_wait_all();                                        // the weight chunk has landed
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core's reads
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int ks = 0; ks < TC_KC / 16; ++ks) {                  // K = 16 per instruction = two core-matrix columns = 256 B
                const uint32_t ko = (uint32_t)ks * 256u;
                const uint64_t a0 = tc_smem_desc(s_a + ko), a1 = tc_smem_desc(s_a + TC_PART_BYTES + ko), a2 = tc_smem_desc(s_a + 2 * TC_PART_BYTES + ko);
                const uint64_t b0 = tc_smem_desc(s_b + ko), b1 = tc_smem_desc(s_b + TC_PART_BYTES + ko), b2 = tc_smem_desc(s_b + 2 * TC_PART_BYTES + ko);
                // the tensor core's fp32 accumulation truncates: the leading term o W0 gets an accumulator of its own (one add per
                // K step), the five corrections — 2^-8 of it and smaller — share the second; the epilogue adds the two
                tc_mma(tmem, a0, b0, TC_IDESC, (c | ks) ? 1u : 0u);
                tc_mma(tmem + 128u, a0, b1, TC_IDESC, (c | ks) ? 1u : 0u);
                tc_mma(tmem + 128u, a1, b0, TC_IDESC, 1u);
                tc_mma(tmem + 128u, a0, b2, TC_IDESC, 1u);
                tc_mma(tmem + 128u, a1, b1, TC_IDESC, 1u);
                tc_mma(tmem + 128u, a2, b0, TC_IDESC, 1u);
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(s_bar) : "memory");
        }
    }
    tc_mbar_wait(s_bar, parity); parity ^= 1u;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- epilogue of layer 1: warp w reads lanes 32 (w & 3) .. + 32 (its rows = r), columns 64 h .. + 64 of both accumulators
    const int q = warp & 3;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    float h1[64];
    {
        uint32_t v[32], u[32];
#pragma unroll
        for (int part = 0; part < 2; ++part) {
            const int col0 = h * 64 + part * 32;
            tc_tmem_ld32(tlane + (uint32_t)col0, v);
            tc_tmem_ld32(tlane + 128u + (uint32_t)col0, u);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const float t = (__uint_as_float(v[i]) + __uint_as_float(u[i])) + bias[col0 + i];
                h1[part * 32 + i] = t > 0.f ? t : t * slope;
            }
        }
    }
    if (MODE == 0) {
        if (row < rows) {
            float4* dst = reinterpret_cast<float4*>(out + row * TC_N + h * 64);
#pragma unroll
            for (int i = 0; i < 16; ++i) dst[i] = make_float4(h1[4 * i], h1[4 * i + 1], h1[4 * i + 2], h1[4 * i + 3]);
        }
    } else {
        // ---- layers 2 and 3: K chunks of 32 (operand parts of 8 KB / 10 KB), one accumulator per layer (48 and 60 adds)
        const uint32_t s_a2 = s_base, s_b2 = s_base + 3 * T2_A_PART;
        const uint32_t a2_row = (uint32_t)((r >> 3) * 512 + (r & 7) * 16);
        auto put_core = [&](int kcol, const float* v8) {                 // 8 consecutive K values of this row -> core column kcol, 3 parts
            uint32_t p0[4], p1[4], p2[4];
#pragma unroll
            for (int e2 = 0; e2 < 4; ++e2) {
                const float a = v8[2 * e2], b = v8[2 * e2 + 1];
                p0[e2] = tc_pack_bf16x2(a, b);
                const float ra = a - __uint_as_float(p0[e2] << 16), rb = b - __uint_as_float(p0[e2] & 0xFFFF0000u);
                p1[e2] = tc_pack_bf16x2(ra, rb);
                p2[e2] = tc_pack_bf16x2(ra - __uint_as_float(p1[e2] << 16), rb - __uint_as_float(p1[e2] & 0xFFFF0000u));
            }
            const uint32_t dst = s_a2 + a2_row + (uint32_t)kcol * 128u;
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(dst), "r"(p0[0]), "r"(p0[1]), "r"(p0[2]), "r"(p0[3]) : "memory");
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(dst + T2_A_PART), "r"(p1[0]), "r"(p1[1]), "r"(p1[2]), "r"(p1[3]) : "memory");
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(dst + 2 * T2_A_PART), "r"(p2[0]), "r"(p2[1]), "r"(p2[2]), "r"(p2[3]) : "memory");
        };
        auto copy_b = [&](const uint4* src, int n16) {                   // the chunk's three weight parts, already in operand layout
#pragma unroll 8
            for (int k = tid; k < n16; k += 256) tc_cp_async16(s_b2 + (uint32_t)k * 16u, src + k);
            tc_cp_async_wait_all();
        };
        auto issue = [&](uint32_t b_part, uint32_t idesc, bool first) {  // one chunk: 2 K steps x 6 products, then commit
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    const uint32_t ko = (uint32_t)ks * 256u;
                    const uint64_t a0 = tc_smem_desc(s_a2 + ko, 512u), a1 = tc_smem_desc(s_a2 + T2_A_PART + ko, 512u), a2 = tc_smem_desc(s_a2 + 2 * T2_A_PART + ko, 512u);
                    const uint64_t b0 = tc_smem_desc(s_b2 + ko, 512u), b1 = tc_smem_desc(s_b2 + b_part + ko, 512u), b2 = tc_smem_desc(s_b2 + 2 * b_part + ko, 512u);
                    tc_mma(tmem, a2, b0, idesc, (first && ks == 0) ? 0u : 1u);     // smallest terms first
                    tc_mma(tmem, a1, b1, idesc, 1u);
                    tc_mma(tmem, a0, b2, idesc, 1u);
                    tc_mma(tmem, a1, b0, idesc, 1u);
                    tc_mma(tmem, a0, b1, idesc, 1u);
                    tc_mma(tmem, a0, b0, idesc, 1u);
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(s_bar) : "memory");
            }
        };
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();                                                  // every thread has read its layer-1 accumulators
        // ---- layer 2: h1 (K = 128: this thread holds columns 64 h .. + 64) x W2 (N = 150 padded to 160)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j > 0) { tc_mbar_wait(s_bar, parity); parity ^= 1u; }
            if (h == (j >> 1)) {
#pragma unroll
                for (int kcol = 0; kcol < 4; ++kcol) put_core(kcol, h1 + 32 * (j & 1) + 8 * kcol);
            }
            copy_b(tw.w2 + (size_t)j * (3 * T2_B160_PART / 16), 3 * T2_B160_PART / 16);
            issue(T2_B160_PART, tc_idesc(160), j == 0);
        }
        tc_mbar_wait(s_bar, parity); parity ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float h2[80];                                                     // columns 80 h .. + 80 of this row
        {
            uint32_t v[16];
#pragma unroll
            for (int part = 0; part < 5; ++part) {
                const int col0 = h * 80 + part * 16;
                tc_tmem_ld16(tlane + (uint32_t)col0, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float t = __uint_as_float(v[i]) + (col0 + i < tw.n2 ? tw.b2[col0 + i] : 0.f);
                    h2[part * 16 + i] = t > 0.f ? t : t * slope;
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        // ---- layer 3: h2 (K = 160: core columns 10 h .. + 10 are this thread's) x W3 (N = 128)
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            if (j > 0) { tc_mbar_wait(s_bar, parity); parity ^= 1u; }
#pragma unroll
            for (int kcol = 0; kcol < 4; ++kcol) {
                const int g = 4 * j + kcol;                               // core column of the whole K
                if (h == (g >= 10 ? 1 : 0)) put_core(kcol, h2 + 8 * (g >= 10 ? g - 10 : g));
            }
            copy_b(tw.w3 + (size_t)j * (3 * T2_A_PART / 16), 3 * T2_A_PART / 16);
            issue(T2_A_PART, tc_idesc(128), j == 0);
        }
        tc_mbar_wait(s_bar, parity); parity ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        float z3[64];                                                     // columns 64 h .. + 64 of this row
        {
            uint32_t v[32];
#pragma unroll
            for (int part = 0; part < 2; ++part) {
                const int col0 = h * 64 + part * 32;
                tc_tmem_ld32(tlane + (uint32_t)col0, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 32; ++i) z3[part * 32 + i] = __uint_as_float(v[i]) + tw.b3[col0 + i];
            }
        }
        if (out && row < rows) {
            float4* dst = reinterpret_cast<float4*>(out + row * TC_N + h * 64);
#pragma unroll
            for (int i = 0; i < 16; ++i) dst[i] = make_float4(z3[4 * i], z3[4 * i + 1], z3[4 * i + 2], z3[4 * i + 3]);
        }
        if (MODE >= 2) {
            // ---- the tail: x = clamp(leaky_relu(z3)); the A + 1 head rows as two 64-term partial sums per row (the two threads
            // of a row meet in shared memory — the operand area is free now); softmax; inverse-CDF sample on one keyed uniform
            // (MODES 2 and 4) or the greedy action (MODES 3 and 5)
            // head weights transposed and zero-padded to [128][12]: the 9 weights of an input are three 16-byte broadcast loads
            float* wsm = reinterpret_cast<float*>(tc_smem);               // [128][12]
            float* partial = wsm + 12 * 128;                              // [128 rows][2 halves][9]
            const int n_out = tw.n_actions + 1;
            for (int k = tid; k < 12 * 128; k += 256) {
                const int i = k / 12, o = k - 12 * i;
                wsm[k] = o < n_out ? tw.w_heads[o * 128 + i] : 0.f;
            }
            __syncthreads();
            float acc[9];
#pragma unroll
            for (int o = 0; o < 9; ++o) acc[o] = 0.f;
#pragma unroll
            for (int i = 0; i < 64; ++i) {
                float v = z3[i];
                v = v > 0.f ? v : v * slope;                              // F.leaky_relu, :92
                v = fminf(fmaxf(v, tw.clamp_lo), tw.clamp_hi);            // torch.clamp(x, -4, 4), :93
                const float4* wrow = reinterpret_cast<const float4*>(wsm + (h * 64 + i) * 12);
                const float4 w0 = wrow[0], w1 = wrow[1], w2 = wrow[2];
                acc[0] = fmaf(v, w0.x, acc[0]); acc[1] = fmaf(v, w0.y, acc[1]); acc[2] = fmaf(v, w0.z, acc[2]); acc[3] = fmaf(v, w0.w, acc[3]);
                acc[4] = fmaf(v, w1.x, acc[4]); acc[5] = fmaf(v, w1.y, acc[5]); acc[6] = fmaf(v, w1.z, acc[6]); acc[7] = fmaf(v, w1.w, acc[7]);
                acc[8] = fmaf(v, w2.x, acc[8]);
            }
#pragma unroll
            for (int o = 0; o < 9; ++o) partial[(r * 2 + h) * 9 + o] = acc[o];
            __syncthreads();
            if (h == 0 && row < rows) {
                const int A = tw.n_actions;
#pragma unroll
                for (int o = 0; o < 9; ++o) acc[o] = o < n_out ? (partial[(r * 2) * 9 + o] + partial[(r * 2 + 1) * 9 + o]) + tw.b_heads[o] : 0.f;
                float mx = -3.4e38f;
#pragma unroll
                for (int o = 0; o < 8; ++o) if (o < A) mx = fmaxf(mx, acc[o]);
                float ex[8], tot = 0.f;
#pragma unroll
                for (int o = 0; o < 8; ++o) { ex[o] = o < A ? expf(acc[o] - mx) : 0.f; tot += ex[o]; }   // F.softmax, :96
                float p_pick = 0.f;
                int pick = A - 1;
                if constexpr (MODE == 2 || MODE == 4) {
                    const uint64_t g = global_env_id(P, row);            // the sampling key: the row's global env id
                    uint32_t c0 = (uint32_t)(g >> 2), c1 = (uint32_t)(g >> 34), c2 = (uint32_t)ctr, c3 = (uint32_t)(ctr >> 32) ^ 0x53414D50u;
#pragma unroll
                    for (int rd = 0; rd < 10; ++rd) {                     // Philox4x32-10 under the sampling seed's round keys
                        const uint64_t p0 = (uint64_t)PHILOX_M0 * c0, p1 = (uint64_t)PHILOX_M1 * c2;
                        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ tw.rk0[rd], n2 = (uint32_t)(p0 >> 32) ^ c3 ^ tw.rk1[rd];
                        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
                    }
                    const uint32_t wd[4] = {c0, c1, c2, c3};
                    const float u = (float)(pick4(wd, (uint32_t)g & 3u) >> 8) * (1.0f / 16777216.0f);
                    const float target = u * tot;
                    float cum = 0.f;
                    bool found = false;
#pragma unroll
                    for (int o = 0; o < 8; ++o) {                         // smallest a with target < e[0] + ... + e[a]
                        cum += ex[o];
                        if (!found && o < A && target < cum) { pick = o; found = true; }
                    }
                } else {
                    // argmax over the LOGITS (two logits may round to one exponential); strict > keeps the lowest index on a tie
                    float best = acc[0];
                    pick = 0;
#pragma unroll
                    for (int o = 1; o < 8; ++o) if (o < A && acc[o] > best) { best = acc[o]; pick = o; }
                }
#pragma unroll
                for (int o = 0; o < 8; ++o) if (o == pick) p_pick = ex[o];
                tw.actions[row] = (uint8_t)pick;
                if (tw.value) tw.value[row] = acc[A < 8 ? A : 8];
                if (tw.logp) tw.logp[row] = logf(p_pick / tot);
                if (tw.probs) {
#pragma unroll
                    for (int o = 0; o < 8; ++o) if (o < A) tw.probs[row * A + o] = ex[o] / tot;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(256u) : "memory");
}

}  // namespace
