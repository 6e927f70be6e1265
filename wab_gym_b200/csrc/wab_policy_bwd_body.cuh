// wab_policy_bwd_body.cuh — the body of wab_policy_bwd_kernel, wab_policy_ppo_bwd_kernel, wab_policy_eval_kernel and
// wab_policy_logits_bwd_kernel and wab_policy_ppo_bwd_population_kernel (wab_policy_bwd.cuh), included inside each. Each
// kernel declares `constexpr BwKind KIND`, its parameters P, food_dim, B, a PpoArgs Q, a ListArgs L and a MemberArgs G;
// KIND selects the row list and the heads block of step 2 (BW_EVAL stops after it), and everything else is shared. A
// fragment rather than a __forceinline__ function: the compiler optimises a device function on its own before inlining
// it, which changes the code of the existing kernels.
    extern __shared__ __align__(1024) uint8_t tc_smem[];
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(tc_smem);
    const uint32_t s_a = s_base + TC_SMEM_A, s_b = s_base + TC_SMEM_B, s_bar = s_base + BW_SMEM_BAR;
    const uint32_t s_m = s_base + BW_SMEM_M, s_n = s_base + BW_SMEM_N;
    uint32_t* rowbits = reinterpret_cast<uint32_t*>(tc_smem + BW_SMEM_BITS);
    float* wsm = reinterpret_cast<float*>(tc_smem + BW_SMEM_WSM);          // head weights transposed, [128][12]
    float* partial = reinterpret_cast<float*>(tc_smem + BW_SMEM_PART);     // [128 rows][2 halves][9]
    float* dhs = reinterpret_cast<float*>(tc_smem + BW_SMEM_DH);           // d heads [128 rows][9]
    float* red = reinterpret_cast<float*>(tc_smem + BW_SMEM_RED);          // [4 warps][160] bias partial sums
    float* part = B.scratch + (size_t)blockIdx.x * BP_BLOCK;
    const int A = B.n_actions, n_out = A + 1;
    constexpr bool LIST = KIND == BW_EVAL || KIND == BW_LOGITS;     // rows by list position, a host count

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"((uint32_t)__cvta_generic_to_shared(&tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(s_bar), "r"(1u) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if constexpr (KIND != BW_EVAL)                                          // the evaluation writes no gradient
        for (int k = tid; k < BP_PARTIAL; k += 256) part[k] = 0.f;
    for (int k = tid; k < 12 * 128; k += 256) {
        const int i = k / 12, o = k - 12 * i;
        wsm[k] = o < n_out ? B.w_heads[o * 128 + i] : 0.f;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_slot;

    const int r = tid & 127, h = tid >> 7, q = warp & 3;
    const uint32_t tlane = tmem + ((uint32_t)(q * 32) << 16);
    const uint32_t* mybits = rowbits + r * TC_ROWBITS_STRIDE;
    const bool noisy = B.noise_scale != 0.f;
    const float scale = B.noise_scale * (1.0f / 16777216.0f), slope = B.slope;
    const uint32_t a_row = (uint32_t)((r >> 3) * 1024 + (r & 7) * 16);
    float* st_h1 = part + BP_H1 + r * 128 + h * 64;                       // this thread's stash: its row, its half
    float* st_h2 = part + BP_H2 + r * 160 + h * 80;
    uint32_t parity = 0;
    long long count = LIST ? L.n_list : (B.d_count ? *B.d_count : (long long)B.n_rows);
    if (!LIST) count = count < 0 ? 0 : (count > (long long)B.n_rows ? (long long)B.n_rows : count);
    if constexpr (KIND == BW_PPO_POP) count = count > G.list_len ? G.list_len : count;   // the member's own list only
    const long long n_tiles = (count + TC_TILE_M - 1) / TC_TILE_M;

    auto wait_mma = [&]() {
        tc_mbar_wait(s_bar, parity); parity ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    // weight-gradient products: M operand (128 rows, K = 128) at s_m, N operand (n rows) at s_n, six products per K step;
    // the tensor core's fp32 accumulation truncates, so the leading product a0 b0 gets an accumulator of its own
    // (column tcol + BW_LEAD) and the five corrections share the one at tcol; returns once the tensor core is done
    auto wg_mma = [&](int n, uint32_t tcol) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t np = (uint32_t)n * 256u, idesc = tc_idesc(n);
#pragma unroll 1
            for (int ks = 0; ks < 8; ++ks) {
                const uint32_t ko = (uint32_t)ks * 256u;
                const uint64_t a0 = tc_smem_desc(s_m + ko, BW_KROW), a1 = tc_smem_desc(s_m + BW_M_PART + ko, BW_KROW), a2 = tc_smem_desc(s_m + 2 * BW_M_PART + ko, BW_KROW);
                const uint64_t b0 = tc_smem_desc(s_n + ko, BW_KROW), b1 = tc_smem_desc(s_n + np + ko, BW_KROW), b2 = tc_smem_desc(s_n + 2 * np + ko, BW_KROW);
                tc_mma(tmem + tcol + BW_LEAD, a0, b0, idesc, ks ? 1u : 0u);
                tc_mma(tmem + tcol, a2, b0, idesc, ks ? 1u : 0u);     // smallest corrections first
                tc_mma(tmem + tcol, a1, b1, idesc, 1u);
                tc_mma(tmem + tcol, a0, b2, idesc, 1u);
                tc_mma(tmem + tcol, a1, b0, idesc, 1u);
                tc_mma(tmem + tcol, a0, b1, idesc, 1u);
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(s_bar) : "memory");
        }
        wait_mma();
    };
    // `cnt` columns of this thread's lane of a wg_mma result at tcol (leading + corrections), added into dst[0 .. cnt)
    // (cnt a multiple of 16)
    auto flush = [&](uint32_t tcol, int cnt, float* dst) {
        uint32_t v[16], u[16];
        for (int c0 = 0; c0 < cnt; c0 += 16) {
            tc_tmem_ld16(tlane + BW_LEAD + tcol + (uint32_t)c0, v);
            tc_tmem_ld16(tlane + tcol + (uint32_t)c0, u);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 16; ++i) dst[c0 + i] += __uint_as_float(v[i]) + __uint_as_float(u[i]);
        }
    };
    // the layer-2 loop of the forward: v (K = 128, this thread's columns 64 h ..) x packed weights with N = 160 -> tensor columns 0 .. 160
    auto put_core = [&](int kcol, const float* v8) {
        uint32_t p0[4], p1[4], p2[4];
#pragma unroll
        for (int e2 = 0; e2 < 4; ++e2) {
            const float a = v8[2 * e2], b = v8[2 * e2 + 1];
            p0[e2] = tc_pack_bf16x2(a, b);
            const float ra = a - __uint_as_float(p0[e2] << 16), rb = b - __uint_as_float(p0[e2] & 0xFFFF0000u);
            p1[e2] = tc_pack_bf16x2(ra, rb);
            p2[e2] = tc_pack_bf16x2(ra - __uint_as_float(p1[e2] << 16), rb - __uint_as_float(p1[e2] & 0xFFFF0000u));
        }
        const uint32_t dst = s_base + (uint32_t)((r >> 3) * 512 + (r & 7) * 16) + (uint32_t)kcol * 128u;
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(dst), "r"(p0[0]), "r"(p0[1]), "r"(p0[2]), "r"(p0[3]) : "memory");
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(dst + T2_A_PART), "r"(p1[0]), "r"(p1[1]), "r"(p1[2]), "r"(p1[3]) : "memory");
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(dst + 2 * T2_A_PART), "r"(p2[0]), "r"(p2[1]), "r"(p2[2]), "r"(p2[3]) : "memory");
    };
    const uint32_t s_b2 = s_base + 3 * T2_A_PART;
    auto copy_b = [&](const uint4* src, int n16) {
#pragma unroll 8
        for (int k = tid; k < n16; k += 256) tc_cp_async16(s_b2 + (uint32_t)k * 16u, src + k);
        tc_cp_async_wait_all();
    };
    // one K chunk of the layer-2 / layer-3 loops. split = false: the forward's single accumulator (the recompute must be
    // bit-identical to it); split = true (the activation gradients): the leading product in its own accumulator at BW_LEAD
    auto issue = [&](uint32_t b_part, uint32_t idesc, bool first, bool split) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
                const uint32_t ko = (uint32_t)ks * 256u;
                const uint64_t a0 = tc_smem_desc(s_base + ko, 512u), a1 = tc_smem_desc(s_base + T2_A_PART + ko, 512u), a2 = tc_smem_desc(s_base + 2 * T2_A_PART + ko, 512u);
                const uint64_t b0 = tc_smem_desc(s_b2 + ko, 512u), b1 = tc_smem_desc(s_b2 + b_part + ko, 512u), b2 = tc_smem_desc(s_b2 + 2 * b_part + ko, 512u);
                tc_mma(tmem, a2, b0, idesc, (first && ks == 0) ? 0u : 1u);
                tc_mma(tmem, a1, b1, idesc, 1u);
                tc_mma(tmem, a0, b2, idesc, 1u);
                tc_mma(tmem, a1, b0, idesc, 1u);
                tc_mma(tmem, a0, b1, idesc, 1u);
                if (split) tc_mma(tmem + BW_LEAD, a0, b0, idesc, (first && ks == 0) ? 0u : 1u);
                else tc_mma(tmem, a0, b0, idesc, 1u);
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(s_bar) : "memory");
        }
    };
    auto dense_128_160 = [&](const float* v64, const uint4* w, float* out80, bool split) {   // K = 128 -> N = 160 (raw sums)
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j > 0) { tc_mbar_wait(s_bar, parity); parity ^= 1u; }
            if (h == (j >> 1)) {
#pragma unroll
                for (int kcol = 0; kcol < 4; ++kcol) put_core(kcol, v64 + 32 * (j & 1) + 8 * kcol);
            }
            copy_b(w + (size_t)j * (3 * T2_B160_PART / 16), 3 * T2_B160_PART / 16);
            issue(T2_B160_PART, tc_idesc(160), j == 0, split);
        }
        wait_mma();
        uint32_t v[16], u[16];
#pragma unroll
        for (int p = 0; p < 5; ++p) {
            tc_tmem_ld16(tlane + (uint32_t)(h * 80 + p * 16), v);
            if (split) tc_tmem_ld16(tlane + BW_LEAD + (uint32_t)(h * 80 + p * 16), u);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 16; ++i) out80[p * 16 + i] = split ? __uint_as_float(u[i]) + __uint_as_float(v[i]) : __uint_as_float(v[i]);
        }
    };
    auto dense_160_128 = [&](const float* v80, const uint4* w, float* out64, bool split) {   // K = 160 -> N = 128 (raw sums)
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 5; ++j) {
            if (j > 0) { tc_mbar_wait(s_bar, parity); parity ^= 1u; }
#pragma unroll
            for (int kcol = 0; kcol < 4; ++kcol) {
                const int g = 4 * j + kcol;
                if (h == (g >= 10 ? 1 : 0)) put_core(kcol, v80 + 8 * (g >= 10 ? g - 10 : g));
            }
            copy_b(w + (size_t)j * (3 * T2_A_PART / 16), 3 * T2_A_PART / 16);
            issue(T2_A_PART, tc_idesc(128), j == 0, split);
        }
        wait_mma();
        uint32_t v[16], u[16];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            tc_tmem_ld16(tlane + (uint32_t)(h * 64 + p * 16), v);
            if (split) tc_tmem_ld16(tlane + BW_LEAD + (uint32_t)(h * 64 + p * 16), u);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int i = 0; i < 16; ++i) out64[p * 16 + i] = split ? __uint_as_float(u[i]) + __uint_as_float(v[i]) : __uint_as_float(v[i]);
        }
    };
    // 32 columns (chunk c, lanes jb .. + 8 of its Philox calls) of this row's input as wab_affine1_tc_kernel generates them
    auto gen_x = [&](int c, uint32_t krow, unsigned long long ctr, float x[4][8]) {
        const int jb = 16 * (c & 1) + 8 * h;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            uint32_t w[4] = {0u, 0u, 0u, 0u};
            if (noisy)
                philox(P, krow, ((uint32_t)(c >> 1) << 24) ^ ((uint32_t)(jb + e) << 16), (uint32_t)ctr,
                       (uint32_t)(ctr >> 32) ^ 0x464C4154u, w);
#pragma unroll
            for (int s = 0; s < 4; ++s) x[s][e] = scale * (float)(w[s] >> 8);
        }
    };

#pragma unroll 1
    for (long long tile = KIND == BW_PPO_POP ? G.cta : blockIdx.x; tile < n_tiles; tile += KIND == BW_PPO_POP ? G.n_cta : gridDim.x) {
        const long long slot = tile * TC_TILE_M + r;
        int64_t flat = slot < count ? (B.rows ? (int64_t)B.rows[slot] : (int64_t)slot) : -1;
        bool valid = flat >= 0 && flat < B.n_rows;                          // a listed row outside [0, T N) contributes nothing,
        if constexpr (KIND == BW_PPO_POP)                                   // nor, in a population, another member's row
            valid = valid && (flat % B.n_envs) / G.member_envs == G.member;
        if (!valid) flat = 0;
        const int64_t step = flat / B.n_envs;
        const uint32_t krow = (uint32_t)global_env_id(P, flat - step * B.n_envs);   // the noise key: the global env id
        const unsigned long long ctr = B.counters[step];
        // ---- the tile's one-hot bit vectors (as wab_affine1_tc_kernel)
        if (tid >= 128) {
            uint32_t* bits = rowbits + r * TC_ROWBITS_STRIDE;
#pragma unroll
            for (int k = 0; k < 16; ++k) bits[k] = 0u;
            if (valid) {
                uint32_t fw[7];
#pragma unroll
                for (int k = 0; k < 7; ++k) fw[k] = reinterpret_cast<const uint32_t*>(B.features)[flat * 7 + k];
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
                if (P.restrict_view) {
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
        // ---- 1. the forward, op for op as wab_affine1_tc_kernel<2>
#pragma unroll 1
        for (int c = 0; c < TC_CHUNKS; ++c) {
            float x[4][8];
            gen_x(c, krow, ctr, x);
            const int jb = 16 * (c & 1) + 8 * h;
            if (c > 0) { tc_mbar_wait(s_bar, parity); parity ^= 1u; }
            {
                const uint4* src = B.w1 + (size_t)c * (3 * TC_PART_BYTES / 16);
#pragma unroll
                for (int k = tid; k < 3 * TC_PART_BYTES / 16; k += 256) tc_cp_async16(s_b + (uint32_t)k * 16u, src + k);
            }
            uint32_t pk[3][4][4];
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const uint32_t ob = (mybits[4 * (c >> 1) + s] >> jb) & 0xFFu;
#pragma unroll
                for (int e2 = 0; e2 < 4; ++e2) {
                    const float oa = (float)((ob >> (2 * e2)) & 1u), obb = (float)((ob >> (2 * e2 + 1)) & 1u);
                    const float na = (oa + x[s][2 * e2]) - oa, nb = (obb + x[s][2 * e2 + 1]) - obb;
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
            tc_cp_async_wait_all();
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int ks = 0; ks < TC_KC / 16; ++ks) {
                    const uint32_t ko = (uint32_t)ks * 256u;
                    const uint64_t a0 = tc_smem_desc(s_a + ko), a1 = tc_smem_desc(s_a + TC_PART_BYTES + ko), a2 = tc_smem_desc(s_a + 2 * TC_PART_BYTES + ko);
                    const uint64_t b0 = tc_smem_desc(s_b + ko), b1 = tc_smem_desc(s_b + TC_PART_BYTES + ko), b2 = tc_smem_desc(s_b + 2 * TC_PART_BYTES + ko);
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
        wait_mma();
        float h1[64];
        {
            uint32_t v[32], u[32];
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                const int col0 = h * 64 + p * 32;
                tc_tmem_ld32(tlane + (uint32_t)col0, v);
                tc_tmem_ld32(tlane + 128u + (uint32_t)col0, u);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float t = (__uint_as_float(v[i]) + __uint_as_float(u[i])) + B.b1[col0 + i];
                    h1[p * 32 + i] = t > 0.f ? t : t * slope;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 64; ++i) st_h1[i] = h1[i];
        float h2[80];
        dense_128_160(h1, B.w2, h2, false);
#pragma unroll
        for (int i = 0; i < 80; ++i) {
            const int col = h * 80 + i;
            const float t = h2[i] + (col < 150 ? B.b2[col] : 0.f);
            h2[i] = t > 0.f ? t : t * slope;
            st_h2[i] = h2[i];
        }
        float z3[64];
        dense_160_128(h2, B.w3, z3, false);
#pragma unroll
        for (int i = 0; i < 64; ++i) z3[i] += B.b3[h * 64 + i];
        // ---- 2. heads, softmax, d heads (the two 64-term halves meet in shared memory, as in the forward)
        {
            float acc[9];
#pragma unroll
            for (int o = 0; o < 9; ++o) acc[o] = 0.f;
#pragma unroll
            for (int i = 0; i < 64; ++i) {
                float v = z3[i];
                v = v > 0.f ? v : v * slope;
                v = fminf(fmaxf(v, B.clamp_lo), B.clamp_hi);
                const float4* wrow = reinterpret_cast<const float4*>(wsm + (h * 64 + i) * 12);
                const float4 w0 = wrow[0], w1 = wrow[1], w2 = wrow[2];
                acc[0] = fmaf(v, w0.x, acc[0]); acc[1] = fmaf(v, w0.y, acc[1]); acc[2] = fmaf(v, w0.z, acc[2]); acc[3] = fmaf(v, w0.w, acc[3]);
                acc[4] = fmaf(v, w1.x, acc[4]); acc[5] = fmaf(v, w1.y, acc[5]); acc[6] = fmaf(v, w1.z, acc[6]); acc[7] = fmaf(v, w1.w, acc[7]);
                acc[8] = fmaf(v, w2.x, acc[8]);
            }
#pragma unroll
            for (int o = 0; o < 9; ++o) partial[(r * 2 + h) * 9 + o] = acc[o];
            __syncthreads();
            if (h == 0) {
#pragma unroll
                for (int o = 0; o < 9; ++o) acc[o] = o < n_out ? (partial[(r * 2) * 9 + o] + partial[(r * 2 + 1) * 9 + o]) + B.b_heads[o] : 0.f;
                if constexpr (LIST) {
                    if constexpr (KIND == BW_EVAL) {                       // logits and value of listed entry m = slot
                        if (slot < count) {
                            const float nan = __int_as_float(0x7FC00000);
#pragma unroll
                            for (int o = 0; o < 8; ++o) if (o < A) L.logits_out[slot * A + o] = valid ? acc[o] : nan;
                            L.value_out[slot] = valid ? acc[A < 8 ? A : 8] : nan;
                        }
                    } else {
#pragma unroll
                        for (int o = 0; o < 9; ++o)                            // d heads as given: d logits, d value
                            dhs[r * 9 + o] = valid && o < n_out ? (o < A ? L.g_logits[slot * A + o] : L.g_value[slot]) : 0.f;
                    }
                } else {
                    float mx = -3.4e38f;
#pragma unroll
                    for (int o = 0; o < 8; ++o) if (o < A) mx = fmaxf(mx, acc[o]);
                    float ex[8], tot = 0.f;
#pragma unroll
                    for (int o = 0; o < 8; ++o) { ex[o] = o < A ? expf(acc[o] - mx) : 0.f; tot += ex[o]; }
                    const int a = valid ? (int)B.actions[flat] : 0;
                    if constexpr (KIND == BW_A2C) {
                        const float gl = valid ? B.g_logp[flat] : 0.f, gv = valid ? B.g_value[flat] : 0.f;
                        float p_pick = 0.f;
#pragma unroll
                        for (int o = 0; o < 8; ++o) if (o == a) p_pick = ex[o];
                        if (valid && B.logp_out) B.logp_out[flat] = logf(p_pick / tot);
                        if (valid && B.value_out) B.value_out[flat] = acc[A < 8 ? A : 8];
#pragma unroll
                        for (int o = 0; o < 9; ++o)                                // d log pi_a / d logit_o = 1[o = a] - p_o; d V = g_value
                            dhs[r * 9 + o] = o < A ? gl * ((o == a ? 1.f : 0.f) - ex[o] / tot) : (o == A ? gv : 0.f);
                    } else {
                        float p_pick = 0.f;
#pragma unroll
                        for (int o = 0; o < 8; ++o) if (o == a) p_pick = ex[o];
                        const float lp = logf(p_pick / tot), value = acc[A < 8 ? A : 8];   // as the forward (and the branch above)
                        // log p_o = (z_o - max) - log sum, never log(p_o): an underflowed p_o would make 0 * log 0 a NaN
                        const float lsum = logf(tot);
                        float ent = 0.f;
#pragma unroll
                        for (int o = 0; o < 8; ++o) if (o < A) ent -= (ex[o] / tot) * ((acc[o] - mx) - lsum);
                        float gl = 0.f, gv = 0.f, wh = 0.f;
                        if (valid) {
                            const float adv = Q.advantage[flat], ratio = expf(lp - Q.logp_old[flat]);
                            const bool clipped = (adv > 0.f && ratio > 1.f + Q.clip_eps) || (adv < 0.f && ratio < 1.f - Q.clip_eps);
                            gl = clipped ? 0.f : (-Q.w_policy * adv) * ratio;
                            gv = Q.w_value * (value - Q.target[flat]);
                            wh = Q.w_entropy;
                            if (B.logp_out) B.logp_out[flat] = lp;
                            if (B.value_out) B.value_out[flat] = value;
                            if (Q.entropy_out) Q.entropy_out[flat] = ent;
                        }
#pragma unroll
                        for (int o = 0; o < 9; ++o) {                          // + d(-w_H H) / d logit_o = w_H p_o (log p_o + H)
                            float d = o < A ? gl * ((o == a ? 1.f : 0.f) - ex[o] / tot) : (o == A ? gv : 0.f);
                            if (o < A && wh != 0.f) d += wh * ((ex[o] / tot) * (((acc[o] - mx) - lsum) + ent));
                            dhs[r * 9 + o] = d;
                        }
                    }
                }
            }
            __syncthreads();
        }
        if constexpr (KIND == BW_EVAL) continue;                           // no gradient: the next tile
        float dh[9];
#pragma unroll
        for (int o = 0; o < 9; ++o) dh[o] = dhs[r * 9 + o];
        // g3 = (W_heads^T d heads) * clamp mask * leaky'(z3); the heads' input act = clamp(leaky(z3)) -> M operand of dW_heads
        float g3[64];
#pragma unroll
        for (int i = 0; i < 64; ++i) {
            const float* wr = wsm + (h * 64 + i) * 12;
            float s = 0.f;
#pragma unroll
            for (int o = 0; o < 9; ++o) s = fmaf(wr[o], dh[o], s);
            const float y = z3[i] > 0.f ? z3[i] : z3[i] * slope;
            const bool pass = y >= B.clamp_lo && y <= B.clamp_hi;
            g3[i] = pass ? (z3[i] > 0.f ? s : s * slope) : 0.f;
            bw_put(s_m, BW_M_PART, h * 64 + i, r, fminf(fmaxf(y, B.clamp_lo), B.clamp_hi));
        }
        // ---- dW_heads^T [in 128][16] = act^T d heads; b_heads = sum of d heads
        if (h == 0) {
#pragma unroll
            for (int o = 0; o < 16; ++o) bw_put(s_n, 16 * 256, o, r, o < 9 ? dh[o] : 0.f);
        }
        wg_mma(16, 0);
        if (h == 0) flush(0, 16, part + BP_WH + (q * 32 + lane) * 16);
        if (tid < 9) {                                                     // 128 terms in order: fp64, or the
            double s = 0.0;                                                // fp32 running sum's rounding dominates
            for (int k = 0; k < 128; ++k) s += (double)dhs[k * 9 + tid];
            part[BP_BH + tid] += (float)s;
        }
        // ---- dW3 [out 128][in 160] = g3^T h2 (two N halves of 80, the half each thread holds); b3
#pragma unroll
        for (int i = 0; i < 64; ++i) bw_put(s_m, BW_M_PART, h * 64 + i, r, g3[i]);
#pragma unroll 1
        for (int nh = 0; nh < 2; ++nh) {
            if (h == nh) {
#pragma unroll
                for (int i = 0; i < 80; ++i) bw_put(s_n, 80 * 256, i, r, st_h2[i]);
            }
            wg_mma(80, 80u * nh);
        }
        flush(80u * h, 80, part + BP_W3 + (q * 32 + lane) * 160 + 80 * h);
        bw_bias_sum(g3, 128, red, part + BP_B3);
        // ---- 3. dh2 = g3 W3 (W3^T packed as a 128 -> 150 layer); g2 = dh2 * leaky'(z2); b2
        float g2[80];
        dense_128_160(g3, B.w3t, g2, true);
#pragma unroll
        for (int i = 0; i < 80; ++i) { const float a2 = st_h2[i]; g2[i] = a2 > 0.f ? g2[i] : g2[i] * slope; }
        bw_bias_sum(g2, 150, red, part + BP_B2);
        // ---- dW2^T [in 128][out 160] = h1^T g2
#pragma unroll
        for (int i = 0; i < 64; ++i) bw_put(s_m, BW_M_PART, h * 64 + i, r, st_h1[i]);
#pragma unroll 1
        for (int nh = 0; nh < 2; ++nh) {
            if (h == nh) {
#pragma unroll
                for (int i = 0; i < 80; ++i) bw_put(s_n, 80 * 256, i, r, g2[i]);
            }
            wg_mma(80, 80u * nh);
        }
        flush(80u * h, 80, part + BP_W2T + (q * 32 + lane) * 160 + 80 * h);
        // ---- dh1 = g2 W2 (W2^T packed as a 150 -> 128 layer); g1 = dh1 * leaky'(z1); b1
        float g1[64];
        dense_160_128(g2, B.w2t, g1, true);
#pragma unroll
        for (int i = 0; i < 64; ++i) { const float a1 = st_h1[i]; g1[i] = a1 > 0.f ? g1[i] : g1[i] * slope; }
        bw_bias_sum(g1, 128, red, part + BP_B1);
        // ---- dW1 [out 128][in] = g1^T x, x regenerated per 64-column slab (the forward's chunk c) as the N operand
#pragma unroll
        for (int i = 0; i < 64; ++i) bw_put(s_m, BW_M_PART, h * 64 + i, r, g1[i]);
#pragma unroll 1
        for (int c = 0; c < TC_CHUNKS; ++c) {
            float x[4][8];
            gen_x(c, krow, ctr, x);
            const int jb = 16 * (c & 1) + 8 * h;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const uint32_t ob = (mybits[4 * (c >> 1) + s] >> jb) & 0xFFu;
#pragma unroll
                for (int e = 0; e < 8; ++e) {                              // slab column 8 (4 h + s) + e: parts o, n0, n1 as the forward's A operand
                    const float o = (float)((ob >> e) & 1u);
                    const float nv = (o + x[s][e]) - o;
                    const __nv_bfloat16 n0 = __float2bfloat16_rn(nv);
                    const __nv_bfloat16 n1 = __float2bfloat16_rn(nv - __bfloat162float(n0));
                    const uint32_t ad = s_n + bw_off(8 * (4 * h + s) + e, r);
                    bw_st16(ad, ((ob >> e) & 1u) * 0x3F80u);
                    bw_st16(ad + 64 * 256, (uint32_t)__bfloat16_as_ushort(n0));
                    bw_st16(ad + 2 * 64 * 256, (uint32_t)__bfloat16_as_ushort(n1));
                }
            }
            wg_mma(64, 0);
            flush(32u * h, 32, part + BP_W1 + (c * 128 + q * 32 + lane) * 64 + 32 * h);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "r"(512u) : "memory");
