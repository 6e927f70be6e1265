// wab_generic.cuh — step / reset kernels for ANY odd viewport up to 31 x 31 and spawn margins 1 and 2 (included by
// wab_kernels.cu). The reference is generic in both (wab_env.py:25-26, :34, :147-148, visible_coords :510-525,
// spawn_wolves :527-576); the fast kernels of wab_kernels.cu are specialised to the default 11 x 11 / margin 1
// geometry (a 121-bit window sliding in four registers). Here one WARP owns one environment:
//   * scalar rules run replicated in every lane (same registers, no divergence: the warp IS the env);
//   * the W x H window is not slid but rebuilt every step from the procedural bush draws — one Philox2x32 call per
//     2 x 2 block, blocks spread over the lanes — minus the depletion log, into a shared-memory bit plane;
//   * wolves (up to 64) sit in shared memory, one lane per wolf for the despawn draw, the chase and the wolf plane;
//   * the two binomial-first sites (spawn ring of (W+2m)(H+2m) - WH cells, wolf init over W*H cells) keep their chosen
//     indices as a short sorted list (the 128-bit mask of wab_core.cuh cannot hold 961 cells);
//   * the observation — 3 x W x H bytes per env at an arbitrary byte offset — goes through the same bit stream and
//     16-byte streaming stores as the fast kernels.
// Rules, draw keys and observation layout are those of wab_core.cuh (and of oracle/keyed_rng.py); results for
// 11 x 11 / margin 1 are identical to the fast kernels (tested).
#pragma once

namespace {

struct GenGeo {
    int32_t W, H, hw, hh, m;      // viewport, half sizes, spawn margin
    int32_t WH, words;            // cells and 32-bit words of a plane
    int32_t ring, bh;             // ring cells, box height H + 2m
    int32_t stream_words, warp_words;   // shared-memory words per warp
};
inline GenGeo make_gen_geo(int W, int H, int m, int wolf_cap) {
    GenGeo g;
    g.W = W; g.H = H; g.hw = W / 2; g.hh = H / 2; g.m = m;
    g.WH = W * H; g.words = (g.WH + 31) / 32;
    g.ring = (W + 2 * m) * (H + 2 * m) - W * H; g.bh = H + 2 * m;
    g.stream_words = (3 * g.WH + 15 + 31) / 32 + 1;
    g.warp_words = 2 * (g.words + 1) + wolf_cap + 32 + g.stream_words;
    return g;
}
constexpr int GEN_WARPS = 4;

struct GenSmem {                  // one warp's slice
    uint32_t* bush;               // [words + 1]  bushes with food in the window (the frame of wab_env.py:266)
    uint32_t* wolf;               // [words + 1]  wolves in the window after the chase (:289)
    uint32_t* wolves;             // [wolf_cap]   packed positions
    uint32_t* chosen;             // [32]         sorted indices of a binomial-first site
    uint32_t* stream;             // [stream_words]
};
__device__ __forceinline__ GenSmem gen_smem(uint32_t* base, const GenGeo& g, int wolf_cap) {
    GenSmem s;
    s.bush = base; s.wolf = s.bush + g.words + 1; s.wolves = s.wolf + g.words + 1; s.chosen = s.wolves + wolf_cap;
    s.stream = s.chosen + 32;
    return s;
}

// bit c of a plane <-> observation cell [i][j] = [hw - (objx - x)][hh - (objy - y)], c = i * H + j (wab_env.py:403-409)
__device__ __forceinline__ int gen_cell_bit(const GenGeo& g, int32_t ddx, int32_t ddy) {   // dd = ostrich - object
    return (ddx + g.hw) * g.H + (ddy + g.hh);
}

// Bushes with food > 0 in the window around (E.x, E.y), as of now: generate_bushes (:613-629) for cells without a record
// is the same draw as for cells seen before (keys do not depend on the turn) minus what was eaten.
__device__ __forceinline__ void gen_window_bushes(const Params& P, const GenGeo& g, const Env& E, const Slots& S,
                                                  uint32_t* bush, int lane) {
    for (int k = lane; k <= g.words; k += 32) bush[k] = 0u;
    __syncwarp();
    if (P.n_bush_thr > 0) {
        const int32_t bx0 = (E.x - g.hw) >> 1, by0 = (E.y - g.hh) >> 1;
        const int nbx = g.hw + 1, nby = g.hh + 1;
        const uint32_t t_hi = P.thr_bush1 >> 16;
        for (int b = lane; b < nbx * nby; b += 32) {
            const int32_t BX = bx0 + b / nby, BY = by0 + b % nby;
            const uint32_t c0 = pack_xy(BX, BY) ^ E.bk_a;
            uint32_t p[2];
            philox2(P, c0, E.bk_b, p);
#pragma unroll
            for (uint32_t l = 0; l < 4u; ++l) {
                const int32_t cx = 2 * BX + (int32_t)(l & 1u), cy = 2 * BY + (int32_t)(l >> 1);
                const int32_t ddx = E.x - cx, ddy = E.y - cy;
                if (ddx < -g.hw || ddx > g.hw || ddy < -g.hh || ddy > g.hh) continue;
                const uint32_t h = ((l & 2u) ? p[1] : p[0]) >> (16u * (l & 1u)) & 0xFFFFu;
                bool on = h > t_hi;
                if (h == t_hi) on = bush_word_rare(c0, E.bk_b, P.rk2[0], l) >= P.thr_bush1;   // 2^-16: the full draw decides
                if (on && E.dep) on = bush_alive(P, E, S, cx, cy) != 0u;
                if (on) {
                    const int c = gen_cell_bit(g, ddx, ddy);
                    atomicOr(bush + (c >> 5), 1u << (c & 31));
                }
            }
        }
    }
    __syncwarp();
}

// ring cell j (oracle/keyed_rng.py ring_index: box-x-major, skipping the view) -> offset from the ostrich
__device__ __forceinline__ void gen_ring_offset(const GenGeo& g, int j, int32_t& dx, int32_t& dy) {
    const int left = g.m * g.bh, mid = g.W * 2 * g.m;
    int bx, by;
    if (j < left) { bx = j / g.bh; by = j % g.bh; }
    else if (j < left + mid) { const int jj = j - left; bx = g.m + jj / (2 * g.m); const int r = jj % (2 * g.m); by = r < g.m ? r : r + g.H; }
    else { const int jj = j - left - mid; bx = g.W + g.m + jj / g.bh; by = jj % g.bh; }
    dx = bx - g.hw - g.m; dy = by - g.hh - g.m;
}

// The chosen indices of a binomial-first site over n cells (the caller saw v >= cdf[0]), ascending, in `chosen`;
// returns their number. Every lane runs the same scalar code; lane 0 keeps the list.
__device__ __forceinline__ int gen_binomial_choose(const Params& P, const Env& E, uint32_t site, uint32_t turn, int32_t n,
                                                   uint64_t v, uint32_t* chosen, int lane) {
    const bool init = site == SITE_INIT;
    int32_t K = 1;
    for (int t = 1; t < 32; ++t) {
        if (v < (init ? P.init_cdf[t] : P.spawn_cdf[t])) break;
        ++K;
    }
    K = K > n ? n : K;
    uint32_t r[4] = {0u, 0u, 0u, 0u};
    for (int32_t i = 0; i < K; ++i) {
        if ((i & 3) == 0) philox(P, E.env_id, E.episode, ctr2(site, turn, 1), (uint32_t)(i >> 2), r);
        int32_t j = (int32_t)(((uint64_t)pick4(r, (uint32_t)i & 3u) * (uint64_t)(uint32_t)(n - i)) >> 32);   // the j-th free index
        int32_t pos = 0;
        for (; pos < i; ++pos) {
            if ((int32_t)chosen[pos] <= j) ++j; else break;
        }
        __syncwarp();
        if (lane == 0) {
            for (int32_t q = i; q > pos; --q) chosen[q] = chosen[q - 1];
            chosen[pos] = (uint32_t)j;
        }
        __syncwarp();
    }
    return K;
}

// 32 bits of a plane starting at bit ls (any sign): bit i of the result = plane bit ls + i, 0 outside [0, WH)
__device__ __forceinline__ uint32_t gen_plane_bits(const uint32_t* plane, int WH, int ls) {
    if (ls <= -32 || ls >= WH) return 0u;
    if (ls < 0) return plane[0] << (-ls);
    const uint32_t v = __funnelshift_r(plane[ls >> 5], plane[(ls >> 5) + 1], (uint32_t)ls & 31u);
    const int valid = WH - ls;
    return valid < 32 ? v & ((1u << valid) - 1u) : v;
}

// Publish the env's observation: 3 * WH bytes at byte offset first_byte of the grids tensor.
__device__ __forceinline__ void gen_emit(const GenGeo& g, const GenSmem& sm, uint8_t* grids, int64_t first_byte, int lane) {
    const int off = (int)(first_byte & 15), centre = g.hw * g.H + g.hh;
    const int nwords = (off + 3 * g.WH + 31) >> 5;
    for (int w = lane; w <= nwords; w += 32) {
        const int s = 32 * w - off;                                  // first env bit of this stream word
        uint32_t v = gen_plane_bits(sm.wolf, g.WH, s) | gen_plane_bits(sm.bush, g.WH, s - g.WH);
        const int o = 2 * g.WH + centre - s;                         // the ostrich plane is its centre cell (:393-410)
        if (o >= 0 && o < 32) v |= 1u << o;
        sm.stream[w] = v;
    }
    __syncwarp();
    stream_flush<false>(sm.stream, nullptr, grids + (first_byte - off), off, off + 3 * g.WH, lane);
    __syncwarp();
}

// reset of this warp's env (wab_env.py:231-248): scalars, window, wolf init; leaves both planes ready for emission
template <bool F64>
__device__ __forceinline__ void gen_reset(const Params& P, const GenGeo& g, Env& E, const Slots& S, const GenSmem& sm,
                                          int lane, uint32_t& overflow) {
    reset_scalars<F64>(P, E);
    gen_window_bushes(P, g, E, S, sm.bush, lane);
    for (int k = lane; k <= g.words; k += 32) sm.wolf[k] = 0u;
    __syncwarp();
    if (P.wolves) {                                                   // initialize_wolves :578-593
        const uint64_t v = binomial_draw(P, E.env_id, E.episode, SITE_INIT, 0u);
        if (v >= P.init_cdf[0]) {
            const int K = gen_binomial_choose(P, E, SITE_INIT, 0u, g.WH, v, sm.chosen, lane);
            for (int i = 0; i < K; ++i) {
                const int c = (int)sm.chosen[i];                      // c = (x + hw) * H + (y + hh)
                const int32_t wx = c / g.H - g.hw, wy = c % g.H - g.hh;
                if (E.nw < (uint32_t)P.wolf_cap) {
                    if (lane == 0) {
                        sm.wolves[E.nw] = pack_xy(wx, wy);
                        const int bit = gen_cell_bit(g, -wx, -wy);
                        sm.wolf[bit >> 5] |= 1u << (bit & 31);
                    }
                    E.nw += 1;
                } else {
                    overflow = 1u;
                }
            }
            __syncwarp();
        }
    }
}

__device__ __forceinline__ void gen_load(const Params& P, const StatePtrs& st, int64_t idx, Env& E, uint32_t* wolves, int lane) {
    const uint32_t pos = st.pos[idx], misc = st.misc[idx], nl = st.nlog[idx];
    E.x = unpack_x(pos); E.y = unpack_y(pos);
    E.food_i = (int32_t)(misc & 0xFFu);
    E.role = (misc >> 8) & 1u; E.status = (misc >> 9) & 3u; E.dep = (misc >> 15) & 1u; E.turn = misc >> 16;
    E.nw = ((misc >> 11) & 15u) | (((nl >> 9) & 7u) << 4);
    E.nlog = nl & 0xFFu; E.stale = (nl >> 8) & 1u;
    E.episode = st.episode[idx]; E.logsig = st.logsig[idx];
    { const uint2 bk = st.bkey[idx]; E.bk_a = bk.x; E.bk_b = bk.y; }
    E.food_f = st.food[idx];
    E.env_id = (uint32_t)global_env_id(P, idx);
    E.m[0] = E.m[1] = E.m[2] = E.m[3] = 0u;
    for (uint32_t k = (uint32_t)lane; k < E.nw; k += 32) wolves[k] = st.wolves[(int64_t)k * st.n + idx];
    __syncwarp();
}
__device__ __forceinline__ void gen_store(const StatePtrs& st, int64_t idx, const Env& E, const uint32_t* wolves, int lane) {
    __syncwarp();
    if (lane == 0) {
        st.pos[idx] = pack_xy(E.x, E.y);
        st.misc[idx] = ((uint32_t)E.food_i & 0xFFu) | (E.role << 8) | (E.status << 9) | ((E.nw & 15u) << 11) | (E.dep << 15) | (E.turn << 16);
        st.episode[idx] = E.episode;
        st.nlog[idx] = (uint16_t)(E.nlog | (E.stale << 8) | ((E.nw >> 4) << 9));
        st.logsig[idx] = E.logsig;
        st.bkey[idx] = make_uint2(E.bk_a, E.bk_b);
        st.food[idx] = E.food_f;
    }
    for (uint32_t k = (uint32_t)lane; k < E.nw; k += 32) st.wolves[(int64_t)k * st.n + idx] = wolves[k];
}

// mask_grid (wab_env.py:344-357): the reference's tile masks are 11 x 11 literals, so restrict_view exists for that size only
__device__ __forceinline__ void gen_view_mask(const Params& P, const GenGeo& g, uint32_t role, const GenSmem& sm, int lane) {
    if (!P.restrict_view || g.WH != CELLS) return;
    if (lane < 4) {
        const uint32_t blind = role == 1u ? P.mask_gath[lane] : P.mask_look[lane];
        sm.wolf[lane] &= ~blind; sm.bush[lane] &= ~blind;
    }
    __syncwarp();
}

__device__ __forceinline__ void gen_write_features(const GenGeo& g, const GenSmem& sm, uint8_t* features, int64_t o,
                                                   uint32_t food_obs, uint32_t role, uint32_t status, int lane) {
    if (!features || g.WH != CELLS || lane != 0) return;
    StepOut O;
    for (int k = 0; k < 4; ++k) { O.wm[k] = sm.wolf[k]; O.bm[k] = sm.bush[k]; }
    O.food_obs = food_obs; O.role = role; O.status = status;
    write_features(features, o, O);
}

// T lockstep steps of every env (wab_env.py:250-342 per step), one warp per env.
template <bool F64>
__global__ void __launch_bounds__(GEN_WARPS * 32) wab_generic_step_kernel(const __grid_constant__ Params P, const StatePtrs st,
                                                                          const GenGeo g, const uint8_t* __restrict__ actions,
                                                                          const int n_steps, const OutPtrs out) {
    extern __shared__ uint32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t idx = (int64_t)blockIdx.x * GEN_WARPS + warp, n = st.n;
    pdl_launch_dependents();
    pdl_wait();
    if (idx >= n) return;
    const GenSmem sm = gen_smem(smem + warp * g.warp_words, g, P.wolf_cap);
    Env E;
    Slots S;
    S.wolves = sm.wolves; S.wstride = 1;
    S.logcell = st.logcell + idx; S.logcnt = st.logcnt + idx; S.lstride = n;
    gen_load(P, st, idx, E, sm.wolves, lane);
    const int centre = g.hw * g.H + g.hh;
    const int64_t obs_bytes = 3 * (int64_t)g.WH;
    uint32_t cnt[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    for (int t = 0; t < n_steps; ++t) {
        const int64_t o = (int64_t)t * n + idx;
        const uint32_t action = actions[o];
        // ---- :251-258 action
        const uint32_t bad = action >= (uint32_t)P.n_actions ? 1u : 0u;
        const uint32_t code = bad ? 0x05u : (uint32_t)(P.act_tbl >> (8 * action)) & 0xFFu;
        const int32_t dx = (int32_t)(code & 3u) - 1, dy = (int32_t)((code >> 2) & 3u) - 1, nrole = (int32_t)((code >> 4) & 3u) - 1;
        E.turn += 1; E.x += dx; E.y += dy;
        if (nrole >= 0) E.role = (uint32_t)nrole;
        uint32_t overflow = 0u;
        // ---- :259, :266 the frame: bushes with food in the window at the new position
        gen_window_bushes(P, g, E, S, sm.bush, lane);
        // ---- :262-264 despawn: one lane per wolf, rank = ordinal among earlier wolves on the same cell
        if (E.nw) {
            uint32_t kept_before = 0, pv[2] = {0u, 0u};
            unsigned keep[2] = {0u, 0u};
            for (int rd = 0; rd < 2; ++rd) {
                const uint32_t k = (uint32_t)(32 * rd + lane);
                bool kp = false;
                if (k < E.nw) {
                    const uint32_t p = sm.wolves[k];
                    uint32_t rank = 0;
                    for (uint32_t q = 0; q < k; ++q) rank += sm.wolves[q] == p ? 1u : 0u;
                    uint32_t w[4];
                    philox(P, E.env_id, E.episode, ctr2(SITE_DESP, E.turn, rank >> 2), p, w);
                    kp = (uint64_t)pick4(w, rank & 3u) >= P.thr_keep;
                    pv[rd] = p;
                }
                keep[rd] = __ballot_sync(FULL, kp);
            }
            __syncwarp();
            for (int rd = 0; rd < 2; ++rd) {
                if ((keep[rd] >> lane) & 1u) sm.wolves[kept_before + (uint32_t)__popc(keep[rd] & ((1u << lane) - 1u))] = pv[rd];
                kept_before += (uint32_t)__popc(keep[rd]);
            }
            E.nw = kept_before;
            __syncwarp();
        }
        const uint32_t status_pre = E.status;
        // ---- :267-297 chase (ties -> x axis), kill on contact, wolf plane after the move
        for (int k = lane; k <= g.words; k += 32) sm.wolf[k] = 0u;
        __syncwarp();
        bool hit = false;
        for (uint32_t k = (uint32_t)lane; k < E.nw; k += 32) {
            const uint32_t p = sm.wolves[k];
            int32_t wx = unpack_x(p), wy = unpack_y(p);
            int32_t ddx = E.x - wx, ddy = E.y - wy;
            if (P.wolves_can_move) {
                const int32_t ax = abs(ddx), ay = abs(ddy);
                const int32_t sx = (ddx > 0) - (ddx < 0), sy = (ddy > 0) - (ddy < 0);
                wx += (ax >= ay) ? sx : 0; wy += (ax < ay) ? sy : 0;
                sm.wolves[k] = pack_xy(wx, wy);
                ddx = E.x - wx; ddy = E.y - wy;
            }
            hit |= ddx == 0 && ddy == 0;
            if (ddx >= -g.hw && ddx <= g.hw && ddy >= -g.hh && ddy <= g.hh) {
                const int c = gen_cell_bit(g, ddx, ddy);
                atomicOr(sm.wolf + (c >> 5), 1u << (c & 31));
            }
        }
        if (__any_sync(FULL, hit) && !P.god_mode) E.status = 2u;
        __syncwarp();
        // ---- :300-313 eat (bush and status as of the frame above)
        uint32_t ate = 0u;
        E.stale = 0u;
        if (((sm.bush[centre >> 5] >> (centre & 31)) & 1u) && (E.role == 1u || P.lookout_only) && status_pre == 0u) {
            ate = 1u;
            if (F64) { double f = E.food_f + P.food_inc; f = f < 0.0 ? 0.0 : f; f = f > 1.0 ? 1.0 : f; E.food_f = f; }
            else { const int32_t f = E.food_i + P.food_int_inc; E.food_i = f > P.food_int_max ? P.food_int_max : f; }
            const uint32_t cell = pack_xy(E.x, E.y);
            const int32_t l = log_find(E, S, cell);
            uint32_t eats = 1u;
            if (l >= 0) {
                eats = (uint32_t)S.logcnt[(int64_t)l * S.lstride] + 1u;
                __syncwarp();
                if (lane == 0) S.logcnt[(int64_t)l * S.lstride] = (uint8_t)eats;
            } else if (E.nlog < (uint32_t)P.log_cap) {
                if (lane == 0) { S.logcell[(int64_t)E.nlog * S.lstride] = cell; S.logcnt[(int64_t)E.nlog * S.lstride] = 1; }
                E.nlog += 1; E.logsig |= cell_sig(cell);
            } else {
                overflow = 1u;
            }
            __syncwarp();
            if (!alive_after(P, bush_word(P, E, E.x, E.y), eats)) { E.dep = 1u; E.stale = 1u; }
        }
        // ---- :316-322 hunger, starvation (overrides killed)
        if (F64) { E.food_f = E.food_f - P.food_dec; if (E.food_f <= 0.0) { E.status = 1u; E.food_f = 0.0; } }
        else { E.food_i -= 1; if (E.food_i <= 0) { E.status = 1u; E.food_i = 0; } }
        // ---- :325-326 spawn_wolves on the ring around the moved ostrich
        if (P.wolves) {
            const uint64_t v = binomial_draw(P, E.env_id, E.episode, SITE_SPAWN, E.turn);
            if (v >= P.spawn_cdf[0]) {
                const int K = gen_binomial_choose(P, E, SITE_SPAWN, E.turn, g.ring, v, sm.chosen, lane);
                for (int i = 0; i < K; ++i) {
                    int32_t ox, oy;
                    gen_ring_offset(g, (int)sm.chosen[i], ox, oy);
                    if (E.nw < (uint32_t)P.wolf_cap) { if (lane == 0) sm.wolves[E.nw] = pack_xy(E.x + ox, E.y + oy); E.nw += 1; }
                    else overflow = 1u;
                }
                __syncwarp();
            }
        }
        // ---- :328-340 reward, done
        uint32_t outcome;
        if (E.status == 0u) outcome = E.turn >= (uint32_t)P.max_turns ? 1u : 0u;
        else outcome = E.status == 1u ? 2u : 3u;
        const uint32_t done = outcome != 0u;
        const float reward = P.reward_table[ate * 4u + outcome];
        const uint32_t info = outcome | (ate << 2) | (bad << 3) | (E.status << 4);
        cnt[WAB_STAT_STEPS] += 1u; cnt[WAB_STAT_EATS] += ate; cnt[WAB_STAT_BAD_ACTIONS] += bad;
        if (done) { cnt[WAB_STAT_EPISODES] += 1u; cnt[outcome == 1u ? WAB_STAT_FINISHED : outcome == 2u ? WAB_STAT_STARVED : WAB_STAT_KILLED] += 1u; }
        if (done && P.auto_reset) gen_reset<F64>(P, g, E, S, sm, lane, overflow);    // VecEnv: the post-reset observation is returned
        cnt[WAB_STAT_OVERFLOWS] += overflow;
        // ---- :342, :359-452 observation
        const uint32_t food_obs = food_observation(P, E, F64);
        gen_view_mask(P, g, E.role, sm, lane);
        if (lane == 0) {
            out.food[o] = (uint8_t)food_obs; out.role[o] = (uint8_t)E.role; out.status[o] = (uint8_t)E.status;
            if (out.reward) out.reward[o] = reward;
            if (out.done) out.done[o] = (uint8_t)done;
            if (out.info) out.info[o] = (uint8_t)info;
        }
        gen_write_features(g, sm, out.features, o, food_obs, E.role, E.status, lane);
        gen_emit(g, sm, out.grids, o * obs_bytes, lane);
    }
    gen_store(st, idx, E, sm.wolves, lane);
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t mine = 0u;
#pragma unroll
    for (int k = 0; k < 8; ++k) mine = lane == k ? cnt[k] : mine;
    if (lane < 8 && mine) st.wstats[gw * 8 + lane] += (unsigned long long)mine;
}

// reset(mask) + fresh observation of every env
template <bool F64>
__global__ void __launch_bounds__(GEN_WARPS * 32) wab_generic_reset_kernel(const __grid_constant__ Params P, const StatePtrs st,
                                                                           const GenGeo g, const uint8_t* __restrict__ mask,
                                                                           const OutPtrs out) {
    extern __shared__ uint32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t idx = (int64_t)blockIdx.x * GEN_WARPS + warp, n = st.n;
    pdl_launch_dependents();
    pdl_wait();
    if (idx >= n) return;
    const GenSmem sm = gen_smem(smem + warp * g.warp_words, g, P.wolf_cap);
    Env E;
    Slots S;
    S.wolves = sm.wolves; S.wstride = 1;
    S.logcell = st.logcell + idx; S.logcnt = st.logcnt + idx; S.lstride = n;
    gen_load(P, st, idx, E, sm.wolves, lane);
    uint32_t overflow = 0u;
    if (mask == nullptr || mask[idx] != 0) {
        gen_reset<F64>(P, g, E, S, sm, lane, overflow);
    } else {                                       // left alone: the observation as last returned
        gen_window_bushes(P, g, E, S, sm.bush, lane);
        const int centre = g.hw * g.H + g.hh;
        for (int k = lane; k <= g.words; k += 32) sm.wolf[k] = 0u;
        __syncwarp();
        if (lane == 0 && E.stale) sm.bush[centre >> 5] |= 1u << (centre & 31);
        for (uint32_t k = (uint32_t)lane; k < E.nw; k += 32) {
            const uint32_t p = sm.wolves[k];
            const int32_t ddx = E.x - unpack_x(p), ddy = E.y - unpack_y(p);
            if (ddx >= -g.hw && ddx <= g.hw && ddy >= -g.hh && ddy <= g.hh) {
                const int c = gen_cell_bit(g, ddx, ddy);
                atomicOr(sm.wolf + (c >> 5), 1u << (c & 31));
            }
        }
        __syncwarp();
    }
    const uint32_t food_obs = food_observation(P, E, F64);
    gen_view_mask(P, g, E.role, sm, lane);
    if (lane == 0) { out.food[idx] = (uint8_t)food_obs; out.role[idx] = (uint8_t)E.role; out.status[idx] = (uint8_t)E.status; }
    gen_write_features(g, sm, out.features, idx, food_obs, E.role, E.status, lane);
    gen_emit(g, sm, out.grids, idx * 3 * (int64_t)g.WH, lane);
    gen_store(st, idx, E, sm.wolves, lane);
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (lane == 0 && overflow) st.wstats[gw * 8 + WAB_STAT_OVERFLOWS] += 1ull;
}

}  // namespace
