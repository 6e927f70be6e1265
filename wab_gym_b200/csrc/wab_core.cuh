// wab_core.cuh — per-environment step logic of the B200 Wolves-and-Bushes simulator.
//
// Everything in this header is one environment's worth of work executed by ONE thread; it is
// written `__host__ __device__` so that tests/hostsim can compile the very same logic with g++ and
// compare it against the oracle without a GPU (a unit test of the kernel logic — the product has no
// CPU path). Warp-cooperative pieces (reset fan-out, observation expansion, coalesced stores) live
// in wab_kernels.cu.
//
// Behaviour follows /root/reference/wab_env.py:250-342 (step), :231-248 (reset), :359-452 (obs);
// each block below cites the lines it implements. Data layout is NOT the reference's:
//   * bushes  : a 121-bit occupancy mask of the 11x11 window (bit i*11+j, [i][j] = [5-dx][5-dy],
//               wab_env.py:403-409) slides with the ostrich; bush values are procedural
//               (food0 = f(keyed draw of the cell)) so only cells that were EATEN need state: a
//               small depletion log (cell, eats). Replaces the ever-growing record frame (:613-629).
//   * wolves  : up to wolf_cap packed (x:i16, y:i16) slots.
//   * food    : integer counter when proven equivalent on the host, else the reference's fp64.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define WAB_HD __host__ __device__ __forceinline__
#define WAB_ROLLED _Pragma("unroll 1")   // rare-path loops stay rolled: the step kernel must fit the instruction cache
#define WAB_HD_RARE __host__ __device__ __noinline__   // rare paths are real calls, kept out of the hot loop's footprint
#else
#define WAB_HD static inline
#define WAB_HD_RARE static
#define WAB_ROLLED
#endif

#ifndef WAB_SLIDE_UNROLL
#define WAB_SLIDE_UNROLL 2
#endif
#ifndef WAB_SPAWN_UNROLL
#define WAB_SPAWN_UNROLL 1
#endif

namespace wab {

// ---- cycle probe of the pipeline kernel's rule warp (a separate build: -DWAB_PIPE_CLOCKS, tools/pipe_clocks.py).
// Lane 0 of each rule warp reads clock64() at the region boundaries of every step and adds the cycles since the previous
// boundary to its warp's row in shared memory; the first active lane of a warp counts each pass through a rare path
// (divergent groups that run it one after another count once each). Without the switch the marks compile to nothing.
enum PipeRegion : int { PC_DRAWS, PC_SLIDE, PC_DEPLOG, PC_DESPAWN, PC_CHASE, PC_EAT, PC_TAIL, PC_RESET, PC_HANDOFF, PC_N };
enum PipePath : int { PP_STEPS, PP_TIE, PP_DEPLOG, PP_WOLVES, PP_EAT, PP_EAT_HIT, PP_SPAWN, PP_RESET, PP_N };
#if defined(WAB_PIPE_CLOCKS) && defined(__CUDACC__)
constexpr int kPcWarps = 8;                     // rule warps per CTA the rows cover (WAB_PIPE_PAIRS <= 8)
__shared__ unsigned long long pc_cyc[kPcWarps][PC_N + 1];   // [PC_N]: clock of the last boundary
__shared__ unsigned int pc_cnt[kPcWarps][PP_N];
__device__ __forceinline__ void pc_mark(int r) {
    const unsigned long long t = clock64();
    if ((threadIdx.x & 31) == 0) {
        unsigned long long* row = pc_cyc[(threadIdx.x >> 5) % kPcWarps];
        row[r] += t - row[PC_N]; row[PC_N] = t;
    }
}
__device__ __forceinline__ void pc_count(int k) {
    if ((int)(threadIdx.x & 31) == __ffs((int)__activemask()) - 1) atomicAdd(&pc_cnt[(threadIdx.x >> 5) % kPcWarps][k], 1u);
}
#endif
#if defined(WAB_PIPE_CLOCKS) && defined(__CUDA_ARCH__)
#define WAB_PC_MARK(r) ::wab::pc_mark(r)
#define WAB_PC_COUNT(k) ::wab::pc_count(k)
#else
#define WAB_PC_MARK(r) ((void)0)
#define WAB_PC_COUNT(k) ((void)0)
#endif

constexpr uint32_t PHILOX_M0 = 0xD2511F53u, PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u, PHILOX_W1 = 0xBB67AE85u;
enum : uint32_t { SITE_BUSH = 1, SITE_INIT = 2, SITE_SPAWN = 3, SITE_DESP = 4, SITE_START = 5 };

constexpr int kSlideUnroll = WAB_SLIDE_UNROLL, kSpawnUnroll = WAB_SPAWN_UNROLL;
constexpr int VIEW = 11, HALF = 5, CELLS = 121, RING = 48;
constexpr int OBS_BYTES = 3 * CELLS;        // 363 bytes per env: wolves, bushes, ostriches
constexpr uint32_t TOP_WORD_MASK = 0x01FFFFFFu;  // 121 = 3*32 + 25

// bit c = 11*i + j.  Column j = 0 -> bits 0,11,...,110 ; column j = 10 -> bits 10,21,...,120
constexpr uint32_t colmask_word(int j, int w) {
    uint32_t m = 0;
    for (int i = 0; i < VIEW; ++i) {
        int c = 11 * i + j;
        if ((c >> 5) == w) m |= 1u << (c & 31);
    }
    return m;
}

template <int J, int W> struct ColMask { static constexpr uint32_t v = colmask_word(J, W); };

// Rule constants + RNG schedule, passed to kernels by value (constant bank).
struct Params {
    uint32_t rk0[10], rk1[10];     // Philox4x32 round keys (key is uniform: the seed)
    uint32_t rk2[10];              // Philox2x32 round keys of the bush draws (key (seed ^ seed >> 32), uniform)
    uint32_t thr_bush1;            // food0 > 0  <=>  word >= thr_bush1   (bush_thr[0])
    uint32_t thr_bush2;            // food0 > 1  <=>  word >= thr_bush2   (bush_thr[1]; only read when n_bush_thr > 1)
    uint64_t spawn_cdf[32], init_cdf[32];  // binomial-first tables: K = #{k : v >= cdf[k]} (oracle/keyed_rng.py)
    uint32_t n_bush_thr;
    uint64_t thr_keep;             // kept <=> word >= thr_keep
    const uint32_t* bush_thr;      // device table, n_bush_thr entries
    uint64_t act_tbl;              // per action a, byte a: (dx+1) | (dy+1)<<2 | (role+1)<<4
    int32_t n_actions, max_turns;
    int32_t food_int_start, food_int_inc, food_int_max;
    int32_t wolf_cap, log_cap;
    uint8_t lookout_only, restrict_view, wolves, wolves_can_move, god_mode, auto_reset;
    int8_t starting_role;
    uint8_t food_random;           // starting_food is None
    double food_start, food_inc, food_dec, food_obs_scale;
    float reward_table[8];
    uint32_t mask_look[4], mask_gath[4];
    uint64_t env_id_base;
    // a handle cut into blocks of c rows (wab_vec_set_replicas / wab_vec_set_blocks), packed into the 8 bytes the field
    // replica_envs always took, so that Params keeps its size and every later argument its constant-bank offset:
    uint32_t replica_envs;         // c, or 0 for a plain handle
    uint32_t block_delta;          // block_stride - c (mod 2^32): -c for replicas (block_stride 0)
};

// The global env id of `row` (< 2^32: wab_vec_set_replicas and wab_vec_set_blocks refuse larger handles), the key of every
// draw the handle makes for it: env_id_base + row, or, on a handle cut into blocks of c rows, env_id_base +
// (row / c) block_stride + row % c = env_id_base + row + (row / c) (block_stride - c): every block repeats the ids of the
// first (replicas, block_stride = 0), or block k holds the ids from env_id_base + k block_stride (blocks). The offset is
// exact in 32 bits (wab_vec_set_blocks refuses a layout whose last id is 2^32 or more past env_id_base). One division and
// one multiply-add inside the branch, as the remainder of replicas took before; a plain handle runs the code it ran.
WAB_HD uint64_t global_env_id(const Params& P, int64_t row) {
    if (P.replica_envs) {
        const uint32_t r = (uint32_t)row;
        return P.env_id_base + (uint64_t)(r + (r / P.replica_envs) * P.block_delta);
    }
    return P.env_id_base + (uint64_t)row;
}

// Registers of one environment.
struct Env {
    int32_t x, y;
    uint32_t turn, role, status, nw, nlog, episode, env_id;
    uint32_t bk_a, bk_b;  // the episode's bush key (words 2, 3 of the START call, oracle/keyed_rng.py)
    uint32_t logsig; // 32-bit Bloom signature of the cells in the depletion log (a clear bit proves absence)
    uint32_t dep;    // 1 once some logged cell has been eaten empty (re-entering cells must consult the log)
    uint32_t stale;  // 1 iff the last step ate the bush under the ostrich empty: that step's observation still
                     // showed it (the frame of :266 predates the eat), and so must a re-emitted one
    uint32_t m[4];   // bush occupancy of the window (food > 0), current
    int32_t food_i;  // INT mode
    double food_f;   // F64 mode
};

// Per-env variable-length storage: element k of this env is base[k * stride].
struct Slots {
    uint32_t* wolves; int32_t wstride;
    uint32_t* logcell; uint8_t* logcnt; int64_t lstride;
};

struct StepOut {
    uint32_t wm[4];   // wolf plane of the observation
    uint32_t bm[4];   // bush plane of the observation (snapshot before eating, wab_env.py:289 vs :312)
    uint32_t food_obs, role, status, done, info;
    float reward;
    uint32_t ate, bad_action, overflow, outcome;
};

// Lanes-per-env cooperation. With LPE > 1 the LPE consecutive lanes of a group hold the SAME env in
// their registers (scalar rules are executed redundantly, which costs nothing when the batch is too
// small to fill the machine) and split the independent Philox calls of a step between them.
template <int LPE> struct Coop { uint32_t sub; uint32_t gmask; };   // sub = lane % LPE, gmask = lanes of the group

template <int LPE>
WAB_HD uint32_t group_or(const Coop<LPE>& c, uint32_t v) {
#if defined(__CUDA_ARCH__)
    if (LPE == 1) return v;
    return __reduce_or_sync(c.gmask, v);
#else
    (void)c;
    return v;
#endif
}

// The lanes of a group run the scalar rules redundantly on ONE env whose wolf slots (shared memory) and depletion
// log (global memory) they share. Stores of a value every lane computes identically are benign; read-modify-write
// updates are not (a lane running ahead would be seen by a lagging one — independent thread scheduling gives no
// lockstep guarantee), so those are made by the group's first lane only, fenced by group_sync on both sides.
template <int LPE>
WAB_HD void group_sync(const Coop<LPE>& c) {
#if defined(__CUDA_ARCH__)
    if (LPE > 1) __syncwarp(c.gmask);
#else
    (void)c;
#endif
}
template <int LPE>
WAB_HD bool group_leader(const Coop<LPE>& c) { return LPE == 1 || c.sub == 0u; }

WAB_HD uint32_t popc32(uint32_t v) {
#if defined(__CUDA_ARCH__)
    return (uint32_t)__popc(v);
#else
    return (uint32_t)__builtin_popcount(v);
#endif
}
WAB_HD uint32_t pack_xy(int32_t x, int32_t y) { return ((uint32_t)x & 0xFFFFu) | ((uint32_t)y << 16); }
WAB_HD int32_t unpack_x(uint32_t p) { return (int32_t)(int16_t)(p & 0xFFFFu); }
WAB_HD int32_t unpack_y(uint32_t p) { return (int32_t)(int16_t)(p >> 16); }

WAB_HD uint32_t fshl(uint32_t lo, uint32_t hi, uint32_t s) {  // upper word of (hi:lo) << s, 0 <= s < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(lo, hi, s);
#else
    return s ? (hi << s) | (lo >> (32 - s)) : hi;
#endif
}
WAB_HD uint32_t fshr(uint32_t lo, uint32_t hi, uint32_t s) {  // lower word of (hi:lo) >> s, 0 <= s < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, s);
#else
    return s ? (lo >> s) | (hi << (32 - s)) : lo;
#endif
}
WAB_HD void shl128(uint32_t* m, uint32_t s) {
    m[3] = fshl(m[2], m[3], s); m[2] = fshl(m[1], m[2], s); m[1] = fshl(m[0], m[1], s); m[0] = m[0] << s;
}
WAB_HD void shr128(uint32_t* m, uint32_t s) {
    m[0] = fshr(m[0], m[1], s); m[1] = fshr(m[1], m[2], s); m[2] = fshr(m[2], m[3], s); m[3] = m[3] >> s;
}
WAB_HD void setbit128(uint32_t* m, int pos, uint32_t on) {
    uint32_t b = on << (pos & 31);
    int w = pos >> 5;
    m[0] |= (w == 0) ? b : 0u; m[1] |= (w == 1) ? b : 0u; m[2] |= (w == 2) ? b : 0u; m[3] |= (w == 3) ? b : 0u;
}

// Philox4x32-10 (Salmon et al. SC'11). Round keys come precomputed from Params.
WAB_HD void philox(const Params& P, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t out[4]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)PHILOX_M0 * c0;
        uint64_t p1 = (uint64_t)PHILOX_M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ P.rk0[r];
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ P.rk1[r];
        c1 = (uint32_t)p1; c3 = (uint32_t)p0; c0 = n0; c2 = n2;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
WAB_HD uint32_t ctr2(uint32_t site, uint32_t turn, uint32_t sub) { return (site << 28) | ((turn & 0xFFFFFu) << 8) | (sub & 0xFFu); }
WAB_HD uint32_t pick4(const uint32_t w[4], uint32_t lane) {
    uint32_t a = (lane & 1u) ? w[1] : w[0];
    uint32_t b = (lane & 1u) ? w[3] : w[2];
    return (lane & 2u) ? b : a;
}

// Philox2x32-10 (same paper; half the multiplies): the bush draws, keyed per episode through the counter.
constexpr uint32_t PHILOX2_M = 0xD256D193u;
WAB_HD void philox2(const Params& P, uint32_t c0, uint32_t c1, uint32_t out[2]) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int r = 0; r < 10; ++r) {
        const uint64_t p = (uint64_t)PHILOX2_M * c0;
        const uint32_t n0 = (uint32_t)(p >> 32) ^ c1 ^ P.rk2[r];
        c1 = (uint32_t)p; c0 = n0;
    }
    out[0] = c0; out[1] = c1;
}
// Cell (x, y) of a 2x2 block owns half-word lane = (x & 1) | (y & 1) << 1 of the block's two words:
// word (y & 1), upper half iff (x & 1).
WAB_HD uint32_t bush_lane(int32_t x, int32_t y) { return ((uint32_t)x & 1u) | (((uint32_t)y & 1u) << 1); }
WAB_HD uint32_t half_sel(uint32_t upper) { return upper ? 0x4432u : 0x4410u; }      // byte-permute selector
WAB_HD uint32_t half_of(uint32_t w, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, sel);
#else
    return sel == 0x4432u ? (w >> 16) : (w & 0xFFFFu);
#endif
}
// Full 32-bit draw of a cell: high half-word from the block call (counter (c0, kb)), low half-word from the
// block's second call (counter (c0, ~kb)); c0 = block ^ ka. Needed for bush VALUES (eating, re-revealing an
// eaten cell) and on a 2^-16 tie of the high half-word with the threshold's, so it is an out-of-line call
// taking scalars only (a Params reference would turn the constant-bank operands into generic loads).
WAB_HD_RARE uint32_t bush_word_rare(uint32_t c0, uint32_t kb, uint32_t key, uint32_t lane) {
    uint32_t a0 = c0, a1 = kb, b0 = c0, b1 = ~kb;
    WAB_ROLLED
    for (int r = 0; r < 10; ++r) {
        const uint64_t pa = (uint64_t)PHILOX2_M * a0, pb = (uint64_t)PHILOX2_M * b0;
        const uint32_t na = (uint32_t)(pa >> 32) ^ a1 ^ key, nb = (uint32_t)(pb >> 32) ^ b1 ^ key;
        a1 = (uint32_t)pa; a0 = na; b1 = (uint32_t)pb; b0 = nb; key += PHILOX_W0;
    }
    const uint32_t sel = half_sel(lane & 1u);
    return (half_of((lane & 2u) ? a1 : a0, sel) << 16) | half_of((lane & 2u) ? b1 : b0, sel);
}
WAB_HD uint32_t bush_word(const Params& P, const Env& E, int32_t x, int32_t y) {
    return bush_word_rare(pack_xy(x >> 1, y >> 1) ^ E.bk_a, E.bk_b, P.rk2[0], bush_lane(x, y));
}
WAB_HD uint32_t cell_sig(uint32_t cell) { return 1u << ((cell * 0x9E3779B1u) >> 27); }
// log slot of a cell, or -1. The signature answers "never eaten here" without touching memory; the
// search runs newest-first because repeated eats hit the most recent entry.
WAB_HD int32_t log_find(const Env& E, const Slots& S, uint32_t cell) {
    if (!(E.logsig & cell_sig(cell))) return -1;
    WAB_ROLLED
    for (uint32_t l = E.nlog; l-- > 0u;)
        if (S.logcell[(int64_t)l * S.lstride] == cell) return (int32_t)l;
    return -1;
}
// A bush whose first-reveal draw is `word` still has food after `eats` eats  <=>  its value
// #{k : thr[k] <= word} exceeds eats  <=>  word >= thr[eats]   (thr ascending; one table load).
WAB_HD uint32_t alive_after(const Params& P, uint32_t word, uint32_t eats) {
    if (eats >= P.n_bush_thr) return 0u;
    if (eats == 1u) return word >= P.thr_bush2 ? 1u : 0u;    // the common case needs no table load
#if defined(__CUDA_ARCH__)
    return word >= __ldg(P.bush_thr + eats) ? 1u : 0u;
#else
    return word >= P.bush_thr[eats] ? 1u : 0u;
#endif
}
// The eat path's form of alive_after: the threshold of `eats` eats is settled on the HIGH half-word of the eaten cell's draw
// (one Philox2x32 call, in line) unless it ties with the threshold's high half (2^-16 per eat: the second call, which
// supplies the low half-word, then runs out of line). Same result as alive_after(P, bush_word(...), eats).
WAB_HD uint32_t eaten_bush_alive(const Params& P, const Env& E, int32_t x, int32_t y, uint32_t eats) {
    if (eats >= P.n_bush_thr) return 0u;
#if defined(__CUDA_ARCH__)
    const uint32_t thr = eats == 1u ? P.thr_bush2 : __ldg(P.bush_thr + eats);
#else
    const uint32_t thr = eats == 1u ? P.thr_bush2 : P.bush_thr[eats];
#endif
    const uint32_t c0 = pack_xy(x >> 1, y >> 1) ^ E.bk_a, lane = bush_lane(x, y);
    uint32_t p[2];
    philox2(P, c0, E.bk_b, p);
    const uint32_t hi = half_of((lane & 2u) ? p[1] : p[0], half_sel(lane & 1u)), thi = thr >> 16;
    if (hi != thi) return hi > thi ? 1u : 0u;
    return bush_word_rare(c0, E.bk_b, P.rk2[0], lane) >= thr ? 1u : 0u;
}
// bush at (x, y) — known to exist at first reveal — still has food? (rare path: only when something was eaten empty)
WAB_HD uint32_t bush_alive(const Params& P, const Env& E, const Slots& S, int32_t x, int32_t y) {
    if (!E.dep) return 1u;                      // nothing has been eaten empty this episode
    int32_t l = log_find(E, S, pack_xy(x, y));
    if (l < 0) return 1u;
    return alive_after(P, bush_word(P, E, x, y), (uint32_t)S.logcnt[(int64_t)l * S.lstride]);
}

// ---- binomial-first sites (oracle/keyed_rng.py): the spawn ring of a step and the window of a reset.
// One Philox call gives a 64-bit draw v; nothing happens iff v < cdf[0] (97.6 % for the ring). Otherwise
// K = #{k : v >= cdf[k]} cells succeed and are chosen one by one among the cells still free.
WAB_HD uint64_t binomial_draw(const Params& P, uint32_t env_id, uint32_t episode, uint32_t site, uint32_t turn) {
    uint32_t w[4];
    philox(P, env_id, episode, ctr2(site, turn, 0), 0u, w);
    return ((uint64_t)w[0] << 32) | (uint64_t)w[1];
}
// Rare path: the chosen cell indices, as a bit mask over n <= 128 cells (bit j of mask[j >> 5]).
// The tables are read straight from the kernel parameters (constant bank), never through a pointer.
WAB_HD void binomial_choose(const Params& P, uint32_t env_id, uint32_t episode, uint32_t site, uint32_t turn,
                                 int32_t n, uint64_t v, uint32_t mask[4]) {
    const bool init = site == SITE_INIT;
    int32_t k = 1;                                       // the caller saw v >= cdf[0]
    WAB_ROLLED
    for (int t = 1; t < 32; ++t) {
        if (v < (init ? P.init_cdf[t] : P.spawn_cdf[t])) break;
        ++k;
    }
    k = k > n ? n : k;
    mask[0] = mask[1] = mask[2] = mask[3] = 0u;
    uint32_t r[4] = {0u, 0u, 0u, 0u};
    WAB_ROLLED
    for (int32_t i = 0; i < k; ++i) {
        if ((i & 3) == 0) philox(P, env_id, episode, ctr2(site, turn, 1), (uint32_t)(i >> 2), r);
        int32_t q = (int32_t)(((uint64_t)pick4(r, (uint32_t)i & 3u) * (uint64_t)(uint32_t)(n - i)) >> 32);
        int32_t j = q;                                    // first choice: the q-th cell is simply cell q
        if (i > 0) {                                      // later choices skip the cells already taken
            j = 0;
            WAB_ROLLED
            for (; j < n; ++j) {
                const uint32_t word = (j >> 5) == 0 ? mask[0] : (j >> 5) == 1 ? mask[1] : (j >> 5) == 2 ? mask[2] : mask[3];
                if (!((word >> (j & 31)) & 1u) && q-- == 0) break;
            }
        }
        setbit128(mask, j, 1u);
    }
}

// 11-bit value with bit g at stride 11 (positions 11*g), as four words.
WAB_HD void spread11(uint32_t v, uint32_t t[4]) {
    t[0] = ((v & 7u) * 0x00100401u) & 0x00400801u;
    t[1] = ((((v >> 3) & 7u) * 0x00100401u) & 0x00400801u) << 1;
    t[2] = ((((v >> 6) & 7u) * 0x00100401u) & 0x00400801u) << 2;
    t[3] = ((((v >> 9) & 3u) * 0x00100401u) & 0x00400801u) << 3;
}

// The line of 11 cells a move by (dx, dy) (one of them non-zero) to (E.x, E.y) reveals, and the 6 bush blocks that hold it:
// slide_window's geometry and block draws for step_draws (slide_window keeps its own copy so that the kernels that do
// not make their draws first compile to the same code as before; test_two_warp_pipeline_* compare the two).
struct SlideLine {
    bool along_y;                 // new row (fixed x) or new column (fixed y)
    int32_t fixed, vmax, vb0, top;
    uint32_t fb, sel0, sel1;
};
WAB_HD SlideLine slide_line(const Env& E, int32_t dx, int32_t dy) {
    SlideLine L;
    L.along_y = (dx != 0);
    L.fixed = L.along_y ? E.x + HALF * dx : E.y + HALF * dy;
    L.vmax = (L.along_y ? E.y : E.x) + HALF;              // cell g of the line has coordinate vmax - g
    L.vb0 = (L.vmax - 10) >> 1;
    L.fb = (uint32_t)L.fixed & 1u;
    // The 6 blocks hold 12 cells, g + 1 = top, top - 1, ..., top - 11 with top = 11 or 12: bit g + 1 of `acc`.
    L.top = L.vmax - 2 * L.vb0 + 1;
    // a line along y meets word e (cell parity e) at half fb; a line along x meets word fb at half e
    L.sel0 = half_sel(L.along_y ? L.fb : 0u); L.sel1 = half_sel(L.along_y ? L.fb : 1u);
    return L;
}
// Block b (0..5) of the line: its two cells' hits (high half-word above the threshold's) at bits top - 2b and
// top - 2b - 1 of `acc`, and whether either high half-word ties with the threshold's.
WAB_HD void slide_block(const Params& P, const Env& E, const SlideLine& L, int b, uint32_t& acc, uint32_t& tie) {
    uint32_t p[2];
    const uint32_t t_hi = P.thr_bush1 >> 16;
    const uint32_t c0 = (L.along_y ? pack_xy(L.fixed >> 1, L.vb0 + b) : pack_xy(L.vb0 + b, L.fixed >> 1)) ^ E.bk_a;
    philox2(P, c0, E.bk_b, p);
    const uint32_t h0 = half_of((L.along_y || !L.fb) ? p[0] : p[1], L.sel0);
    const uint32_t h1 = half_of((L.along_y || L.fb) ? p[1] : p[0], L.sel1);
    const uint32_t bit = 1u << (L.top - 2 * b);
    acc |= (h0 > t_hi ? bit : 0u) | (h1 > t_hi ? (bit >> 1) : 0u);
    tie |= (h0 == t_hi ? 1u : 0u) | (h1 == t_hi ? 1u : 0u);
}

// The keyed draws of one step that depend only on the env's state before the step and its action (env_step_pipe):
// this lane's slide blocks and the spawn draw.
struct StepDraws {
    uint32_t acc, tie;   // slide_block over this lane's blocks b = sub, sub + LPE, ... < 6
    uint64_t spawn;      // binomial_draw of SITE_SPAWN at the step's turn
};

// Slide the window after the ostrich moved by (dx, dy) (one of them non-zero) to (E.x, E.y) and
// reveal the 11 new cells: generate_bushes, wab_env.py:613-629, for cells without a record; cells
// seen before get the same draw (keys do not depend on the turn) minus what was eaten.
template <int LPE>
WAB_HD void slide_window(const Params& P, Env& E, const Slots& S, int32_t dx, int32_t dy, const Coop<LPE>& coop) {
    // drop the column that would wrap into the neighbouring row, then shift by 11*dx + dy
    if (dy > 0) {
        E.m[0] &= ~ColMask<10, 0>::v; E.m[1] &= ~ColMask<10, 1>::v; E.m[2] &= ~ColMask<10, 2>::v; E.m[3] &= ~ColMask<10, 3>::v;
    }
    if (dy < 0) {
        E.m[0] &= ~ColMask<0, 0>::v; E.m[1] &= ~ColMask<0, 1>::v; E.m[2] &= ~ColMask<0, 2>::v; E.m[3] &= ~ColMask<0, 3>::v;
    }
    int32_t s = 11 * dx + dy;
    shl128(E.m, (uint32_t)(s > 0 ? s : 0));
    shr128(E.m, (uint32_t)(s < 0 ? -s : 0));
    E.m[3] &= TOP_WORD_MASK;

    const bool along_y = (dx != 0);                       // new row (fixed x) or new column (fixed y)
    const int32_t fixed = along_y ? E.x + HALF * dx : E.y + HALF * dy;
    const int32_t vmax = (along_y ? E.y : E.x) + HALF;    // cell g of the line has coordinate vmax - g
    const int32_t vb0 = (vmax - 10) >> 1;
    const uint32_t fb = (uint32_t)fixed & 1u;
    // The 6 blocks hold 12 cells, g + 1 = top, top - 1, ..., top - 11 with top = 11 or 12: bit g + 1 of `acc`.
    const int32_t top = vmax - 2 * vb0 + 1;
    const uint32_t t_hi = P.thr_bush1 >> 16;
    // a line along y meets word e (cell parity e) at half fb; a line along x meets word fb at half e
    const uint32_t sel0 = half_sel(along_y ? fb : 0u), sel1 = half_sel(along_y ? fb : 1u);
    uint32_t acc = 0, tie = 0;
    if (P.n_bush_thr > 0) {
#if defined(__CUDA_ARCH__)
#pragma unroll kSlideUnroll
#endif
        for (int b = (int)coop.sub; b < 6; b += LPE) {   // slide_block, written out
            uint32_t p[2];
            const uint32_t c0 = (along_y ? pack_xy(fixed >> 1, vb0 + b) : pack_xy(vb0 + b, fixed >> 1)) ^ E.bk_a;
            philox2(P, c0, E.bk_b, p);
            const uint32_t h0 = half_of((along_y || !fb) ? p[0] : p[1], sel0);
            const uint32_t h1 = half_of((along_y || fb) ? p[1] : p[0], sel1);
            const uint32_t bit = 1u << (top - 2 * b);
            acc |= (h0 > t_hi ? bit : 0u) | (h1 > t_hi ? (bit >> 1) : 0u);
            tie |= (h0 == t_hi ? 1u : 0u) | (h1 == t_hi ? 1u : 0u);
        }
        if (tie) {                 // 2^-15 per block: settle this lane's cells on their full 32-bit draws
            acc = 0;
            WAB_ROLLED
            for (int b = (int)coop.sub; b < 6; b += LPE) {
                const uint32_t c0 = (along_y ? pack_xy(fixed >> 1, vb0 + b) : pack_xy(vb0 + b, fixed >> 1)) ^ E.bk_a;
                WAB_ROLLED
                for (uint32_t e = 0; e < 2u; ++e) {
                    const uint32_t lane = along_y ? (fb | (e << 1)) : (e | (fb << 1));
                    if (bush_word_rare(c0, E.bk_b, P.rk2[0], lane) >= P.thr_bush1) acc |= 1u << (top - 2 * b - (int32_t)e);
                }
            }
        }
        acc &= 0xFFEu;             // cells g = 0..10
        if (E.dep) {               // something was eaten empty this episode: revealed cells consult the log
            uint32_t bits = acc;
            WAB_ROLLED
            while (bits) {
#if defined(__CUDA_ARCH__)
                const int k = __ffs((int)bits) - 1;
#else
                const int k = __builtin_ctz(bits);
#endif
                bits &= bits - 1u;
                const int32_t v = vmax - (k - 1);
                if (!(along_y ? bush_alive(P, E, S, fixed, v) : bush_alive(P, E, S, v, fixed))) acc &= ~(1u << k);
            }
        }
    }
    uint32_t line = acc >> 1;
    line = group_or(coop, line);
    if (along_y) {                                // row i = 0 (dx > 0) or i = 10 (dx < 0): bits 11*i + g
        E.m[0] |= (dx > 0) ? line : 0u;
        E.m[3] |= (dx < 0) ? (line << 14) : 0u;   // 110 = 96 + 14
    } else {                                      // column j = 0 (dy > 0) or j = 10 (dy < 0): bits 11*g + j
        uint32_t t[4];
        spread11(line, t);
        shl128(t, dy < 0 ? 10u : 0u);
        E.m[0] |= t[0]; E.m[1] |= t[1]; E.m[2] |= t[2]; E.m[3] |= t[3];
    }
}

// ring cell j (oracle/keyed_rng.py ring_index) -> offset from the ostrich
WAB_HD void ring_offset(int j, int32_t& dx, int32_t& dy) {
    int bx, by;
    if (j < 13) { bx = 0; by = j; }
    else if (j < 35) { bx = 1 + ((j - 13) >> 1); by = ((j - 13) & 1) ? 12 : 0; }
    else { bx = 12; by = j - 35; }
    dx = bx - 6; dy = by - 6;
}

WAB_HD uint32_t food_observation(const Params& P, const Env& E, bool f64) {
    if (!f64) return (uint32_t)E.food_i;
#if defined(__CUDA_ARCH__)
    return (uint32_t)(int32_t)ceil(__dmul_rn(E.food_f, P.food_obs_scale));   // wab_env.py:452
#else
    return (uint32_t)(int32_t)__builtin_ceil(E.food_f * P.food_obs_scale);
#endif
}

// wolf plane from the current wolf slots (wab_env.py:412-428)
WAB_HD void wolf_plane(const Env& E, const Slots& S, uint32_t wm[4]) {
    wm[0] = wm[1] = wm[2] = wm[3] = 0u;
    WAB_ROLLED
    for (uint32_t k = 0; k < E.nw; ++k) {
        uint32_t p = S.wolves[(int32_t)k * S.wstride];
        int32_t ddx = E.x - unpack_x(p), ddy = E.y - unpack_y(p);
        if (ddx >= -HALF && ddx <= HALF && ddy >= -HALF && ddy <= HALF)
            setbit128(wm, 11 * (ddx + HALF) + (ddy + HALF), 1u);
    }
}

// The draws of StepDraws for the step whose action has just moved the ostrich to (E.x, E.y) and advanced E.turn.
// Straight-line code on every lane — lanes without a block (sub >= 6) draw a harmless duplicate and mask it out — so the
// independent Philox chains interleave with each other instead of running one after another. (The despawn draws were
// made here too, wolf k = sub, and measured 6 % slower: they cost a Philox4x32 on every step, wolves or not.)
template <int LPE>
WAB_HD StepDraws step_draws(const Params& P, const Env& E, int32_t dx, int32_t dy, const Coop<LPE>& coop) {
    StepDraws D;
    D.spawn = binomial_draw(P, E.env_id, E.episode, SITE_SPAWN, E.turn);
    D.acc = 0u; D.tie = 0u;
    const SlideLine L = slide_line(E, dx, dy);
    constexpr int NB = (6 + LPE - 1) / LPE;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < NB; ++j) {
        const int b = (int)coop.sub + j * LPE;
        uint32_t acc = 0u, tie = 0u;
        slide_block(P, E, L, b < 6 ? b : 5, acc, tie);
        D.acc |= b < 6 ? acc : 0u; D.tie |= b < 6 ? tie : 0u;
    }
    return D;
}

// One step of one environment: wab_env.py:250-342 up to (not including) auto-reset and the
// observation stores. `F64` selects the reference's fp64 food arithmetic.
template <bool F64, int LPE>
WAB_HD void env_step(const Params& P, Env& E, const Slots& S, uint32_t action, StepOut& O, const Coop<LPE>& coop) {
    // ---- :251-258 action
    O.bad_action = (action >= (uint32_t)P.n_actions) ? 1u : 0u;
    const uint32_t code = O.bad_action ? 0x05u /* dx=0, dy=0, keep */ : (uint32_t)(P.act_tbl >> (8 * action)) & 0xFFu;
    const int32_t dx = (int32_t)(code & 3u) - 1, dy = (int32_t)((code >> 2) & 3u) - 1;
    const int32_t nrole = (int32_t)((code >> 4) & 3u) - 1;
    E.turn += 1;                                   // :252
    E.x += dx; E.y += dy;                          // :255-256
    if (nrole >= 0) E.role = (uint32_t)nrole;      // :257-258
    O.overflow = 0;

    // ---- :259 generate_bushes for the newly visible line
    if (dx != 0 || dy != 0) slide_window<LPE>(P, E, S, dx, dy, coop);

    // ---- :262-264 despawn (keep iff U > chance). rank = ordinal among earlier wolves on the cell.
    if (E.nw) {
        uint32_t kept = 0;
        uint64_t keepmask = 0;                         // wolf_cap <= 64
        WAB_ROLLED
        for (uint32_t k = 0; k < E.nw; ++k) {
            const uint32_t p = S.wolves[(int32_t)k * S.wstride];
            uint32_t rank = 0;
            WAB_ROLLED
            for (uint32_t q = 0; q < k; ++q) rank += (S.wolves[(int32_t)q * S.wstride] == p) ? 1u : 0u;
            uint32_t w[4];
            philox(P, E.env_id, E.episode, ctr2(SITE_DESP, E.turn, rank >> 2), p, w);
            if ((uint64_t)pick4(w, rank & 3u) >= P.thr_keep) keepmask |= 1ull << k;
        }
        group_sync(coop);                       // every lane of the group has read the slots
        if (group_leader(coop)) {
            WAB_ROLLED
            for (uint32_t k = 0; k < E.nw; ++k)
                if ((keepmask >> k) & 1ull) {
                    S.wolves[(int32_t)kept * S.wstride] = S.wolves[(int32_t)k * S.wstride];
                    ++kept;
                }
        }
        group_sync(coop);
        E.nw = popc32((uint32_t)keepmask) + popc32((uint32_t)(keepmask >> 32));
    }

    // ---- :266 the frame the rest of the step reads: bushes with food > 0, ostrich status
    O.bm[0] = E.m[0]; O.bm[1] = E.m[1]; O.bm[2] = E.m[2]; O.bm[3] = E.m[3];
    const uint32_t status_pre = E.status;

    // ---- :267-297 wolves chase (ties -> x axis), kill on contact; wolf plane after the move (:289)
    O.wm[0] = O.wm[1] = O.wm[2] = O.wm[3] = 0u;
    WAB_ROLLED
    for (uint32_t k = 0; k < E.nw; ++k) {
        const uint32_t p = S.wolves[(int32_t)k * S.wstride];
        int32_t wx = unpack_x(p), wy = unpack_y(p);
        int32_t ddx = E.x - wx, ddy = E.y - wy;                                  // :59-60
        if (P.wolves_can_move) {
            const int32_t ax = ddx < 0 ? -ddx : ddx, ay = ddy < 0 ? -ddy : ddy;
            const int32_t sx = (ddx > 0) - (ddx < 0), sy = (ddy > 0) - (ddy < 0);
            wx += (ax >= ay) ? sx : 0;                                           // :278-280
            wy += (ax < ay) ? sy : 0;                                            // :281-283
            group_sync(coop);                                                    // all lanes hold the old position
            if (group_leader(coop)) S.wolves[(int32_t)k * S.wstride] = pack_xy(wx, wy);   // :285-286
            ddx = E.x - wx; ddy = E.y - wy;
        }
        if (ddx == 0 && ddy == 0 && !P.god_mode) E.status = 2u;                  // :292-297
        if (ddx >= -HALF && ddx <= HALF && ddy >= -HALF && ddy <= HALF)          // :416-427
            setbit128(O.wm, 11 * (ddx + HALF) + (ddy + HALF), 1u);
    }
    if (E.nw && P.wolves_can_move) group_sync(coop);                             // moved positions published to the group

    // ---- :300-313 eat (bush and status as of the frame above; role is fresh)
    O.ate = 0;
    E.stale = 0u;
    if (((O.bm[1] >> 28) & 1u) && (E.role == 1u || P.lookout_only) && status_pre == 0u) {   // bit 60 = [5][5]
        O.ate = 1u;
        if (F64) {
            double f = E.food_f + P.food_inc;                                    // :307-309
            f = f < 0.0 ? 0.0 : f; f = f > 1.0 ? 1.0 : f;                        // :310
            E.food_f = f;
        } else {
            int32_t f = E.food_i + P.food_int_inc;
            E.food_i = f > P.food_int_max ? P.food_int_max : f;
        }
        // bush.food -= 1 (:312): count the eat; the cell disappears when eats == its first-reveal value
        const uint32_t cell = pack_xy(E.x, E.y);
        int32_t l = log_find(E, S, cell);
        uint32_t eats;
        if (l >= 0) {
            eats = (uint32_t)S.logcnt[(int64_t)l * S.lstride] + 1u;
            group_sync(coop);                      // every lane of the group has read the old count
            if (group_leader(coop)) S.logcnt[(int64_t)l * S.lstride] = (uint8_t)eats;
            group_sync(coop);
        } else if (E.nlog < (uint32_t)P.log_cap) {
            eats = 1u;
            S.logcell[(int64_t)E.nlog * S.lstride] = cell;
            S.logcnt[(int64_t)E.nlog * S.lstride] = 1;
            E.nlog += 1;
            E.logsig |= cell_sig(cell);
        } else {
            eats = 1u; O.overflow = 1u;            // counted, never silent (WAB_STAT_OVERFLOWS)
        }
        const uint32_t still = eaten_bush_alive(P, E, E.x, E.y, eats);
        if (!still) { E.m[1] &= ~(1u << 28); E.dep = 1u; E.stale = 1u; }
    }

    // ---- :316-322 hunger, starvation (overrides killed)
    if (F64) {
        E.food_f = E.food_f - P.food_dec;
        if (E.food_f <= 0.0) { E.status = 1u; E.food_f = 0.0; }
    } else {
        E.food_i -= 1;
        if (E.food_i <= 0) { E.status = 1u; E.food_i = 0; }
    }

    // ---- :325-326 spawn_wolves on the 48 ring cells around the moved ostrich: one binomial-first draw
    if (P.wolves) {
        const uint64_t v = binomial_draw(P, E.env_id, E.episode, SITE_SPAWN, E.turn);
        if (v >= P.spawn_cdf[0]) {                 // rare (2.4 % of steps): at least one wolf appears
            uint32_t chosen[4];
            binomial_choose(P, E.env_id, E.episode, SITE_SPAWN, E.turn, RING, v, chosen);
            WAB_ROLLED
            for (int w = 0; w < 2; ++w) {                                         // :571-574, ring order
                uint32_t bits = w ? chosen[1] : chosen[0];
                WAB_ROLLED
                while (bits) {
#if defined(__CUDA_ARCH__)
                    const int j = 32 * w + __ffs((int)bits) - 1;
#else
                    const int j = 32 * w + __builtin_ctz(bits);
#endif
                    bits &= bits - 1u;
                    int32_t ox, oy;
                    ring_offset(j, ox, oy);
                    if (E.nw < (uint32_t)P.wolf_cap) {
                        S.wolves[(int32_t)E.nw * S.wstride] = pack_xy(E.x + ox, E.y + oy);
                        E.nw += 1;
                    } else {
                        O.overflow = 1u;
                    }
                }
            }
        }
    }
    // ---- :328-340 reward, done
    uint32_t outcome;
    if (E.status == 0u) outcome = (E.turn >= (uint32_t)P.max_turns) ? 1u : 0u;
    else outcome = (E.status == 1u) ? 2u : 3u;
    O.outcome = outcome;
    O.done = outcome != 0u;
    O.reward = P.reward_table[O.ate * 4u + outcome];
    O.info = outcome | (O.ate << 2) | (O.bad_action << 3) | (E.status << 4);

    // ---- :342, :387-391, :450-452 scalar observation (fresh)
    O.food_obs = food_observation(P, E, F64);
    O.role = E.role;
    O.status = E.status;
}

// OR over the LPE lanes of a group as a butterfly; the whole warp must be converged here (env_step_pipe).
template <int LPE>
WAB_HD uint32_t group_or_converged(uint32_t v) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int o = 1; o < LPE; o <<= 1) v |= __shfl_xor_sync(0xFFFFFFFFu, v, o);
#endif
    return v;
}
// A warp-uniform test: every lane takes the branch if any lane needs it, so the warp never splits on it.
#if defined(__CUDA_ARCH__)
#define WAB_ANY(p) __any_sync(0xFFFFFFFFu, (p))
#else
#define WAB_ANY(p) (p)
#endif

// slide_window's settling of a revealed line on full 32-bit draws, for a lane whose blocks had a tie (2^-15 per block).
template <int LPE>
WAB_HD uint32_t slide_settle(const Params& P, const Env& E, const SlideLine& L, uint32_t sub) {
    uint32_t acc = 0u;
    WAB_ROLLED
    for (int b = (int)sub; b < 6; b += LPE) {
        const uint32_t c0 = (L.along_y ? pack_xy(L.fixed >> 1, L.vb0 + b) : pack_xy(L.vb0 + b, L.fixed >> 1)) ^ E.bk_a;
        WAB_ROLLED
        for (uint32_t e = 0; e < 2u; ++e) {
            const uint32_t lane = L.along_y ? (L.fb | (e << 1)) : (e | (L.fb << 1));
            if (bush_word_rare(c0, E.bk_b, P.rk2[0], lane) >= P.thr_bush1) acc |= 1u << (L.top - 2 * b - (int32_t)e);
        }
    }
    return acc;
}

// env_step for the pipeline kernel's rule warp, with the same results. Every lane of the warp calls it, converged; lanes
// whose env does not exist (`active` false, the ragged last warp) step a neutral Env that never eats or spawns and whose
// results the caller drops. The step's keyed draws are made first (step_draws), and the common step is straight-line code:
// every env slides (a stay is a shift by 0 and an empty deposit), both deposit forms are computed and selected, and the
// group's OR of the revealed line is a butterfly. Each rare path (a tie of a revealed block, the depletion log of an env
// that has eaten a bush empty, wolves, an eat, a spawn) is entered through one warp-uniform test, so the warp never splits
// on it: inside, each env is predicated as in env_step, and the warp runs the path once whichever of its envs need it.
template <bool F64, int LPE>
WAB_HD void env_step_pipe(const Params& P, Env& E, const Slots& S, uint32_t action, StepOut& O, const Coop<LPE>& coop,
                          bool active) {
    // ---- :251-258 action
    O.bad_action = (action >= (uint32_t)P.n_actions) ? 1u : 0u;
    const uint32_t code = O.bad_action ? 0x05u /* dx=0, dy=0, keep */ : (uint32_t)(P.act_tbl >> (8 * action)) & 0xFFu;
    const int32_t dx = (int32_t)(code & 3u) - 1, dy = (int32_t)((code >> 2) & 3u) - 1;
    const int32_t nrole = (int32_t)((code >> 4) & 3u) - 1;
    E.turn += 1;                                   // :252
    E.x += dx; E.y += dy;                          // :255-256
    E.role = nrole >= 0 ? (uint32_t)nrole : E.role;   // :257-258
    O.overflow = 0;
    const StepDraws D = step_draws<LPE>(P, E, dx, dy, coop);
    WAB_PC_MARK(PC_DRAWS);

    // ---- :259 generate_bushes for the newly visible line (slide_window)
    const uint32_t d0 = dy > 0 ? ColMask<10, 0>::v : dy < 0 ? ColMask<0, 0>::v : 0u;
    const uint32_t d1 = dy > 0 ? ColMask<10, 1>::v : dy < 0 ? ColMask<0, 1>::v : 0u;
    const uint32_t d2 = dy > 0 ? ColMask<10, 2>::v : dy < 0 ? ColMask<0, 2>::v : 0u;
    const uint32_t d3 = dy > 0 ? ColMask<10, 3>::v : dy < 0 ? ColMask<0, 3>::v : 0u;
    E.m[0] &= ~d0; E.m[1] &= ~d1; E.m[2] &= ~d2; E.m[3] &= ~d3;
    const int32_t s = 11 * dx + dy;
    shl128(E.m, (uint32_t)(s > 0 ? s : 0));
    shr128(E.m, (uint32_t)(s < 0 ? -s : 0));
    E.m[3] &= TOP_WORD_MASK;
    const bool reveal = (dx != 0 || dy != 0) && P.n_bush_thr > 0;
    const SlideLine L = slide_line(E, dx, dy);
    uint32_t acc = reveal ? D.acc : 0u;
    const uint32_t tie = reveal ? D.tie : 0u;
    if (WAB_ANY(tie != 0u)) {
        WAB_PC_COUNT(PP_TIE);
        if (tie) acc = slide_settle<LPE>(P, E, L, coop.sub);
    }
    acc &= 0xFFEu;                                 // cells g = 0..10
    WAB_PC_MARK(PC_SLIDE);
    if (WAB_ANY(E.dep && acc)) {                   // something was eaten empty this episode: revealed cells consult the log
        WAB_PC_COUNT(PP_DEPLOG);
        uint32_t bits = E.dep ? acc : 0u;
        WAB_ROLLED
        while (bits) {
#if defined(__CUDA_ARCH__)
            const int k = __ffs((int)bits) - 1;
#else
            const int k = __builtin_ctz(bits);
#endif
            bits &= bits - 1u;
            const int32_t v = L.vmax - (k - 1);
            if (!(L.along_y ? bush_alive(P, E, S, L.fixed, v) : bush_alive(P, E, S, v, L.fixed))) acc &= ~(1u << k);
        }
    }
    WAB_PC_MARK(PC_DEPLOG);
    {
        const uint32_t line = group_or_converged<LPE>(acc >> 1);
        uint32_t t[4];                             // column j = 0 (dy > 0) or j = 10 (dy < 0): bits 11*g + j
        spread11(line, t);
        shl128(t, dy < 0 ? 10u : 0u);
        const bool along_y = dx != 0;              // row i = 0 (dx > 0) or i = 10 (dx < 0): bits 11*i + g
        E.m[0] |= along_y ? (dx > 0 ? line : 0u) : t[0];
        E.m[1] |= along_y ? 0u : t[1];
        E.m[2] |= along_y ? 0u : t[2];
        E.m[3] |= along_y ? (dx < 0 ? (line << 14) : 0u) : t[3];   // 110 = 96 + 14
    }
    WAB_PC_MARK(PC_SLIDE);

    // ---- :262-264 despawn (keep iff U > chance). rank = ordinal among earlier wolves on the cell.
    const bool any_wolf = WAB_ANY(E.nw != 0u);
    if (any_wolf) {
        WAB_PC_COUNT(PP_WOLVES);
        if (E.nw) {
            uint32_t kept = 0;
            uint64_t keepmask = 0;                         // wolf_cap <= 64
            WAB_ROLLED
            for (uint32_t k = 0; k < E.nw; ++k) {
                const uint32_t p = S.wolves[(int32_t)k * S.wstride];
                uint32_t rank = 0;
                WAB_ROLLED
                for (uint32_t q = 0; q < k; ++q) rank += (S.wolves[(int32_t)q * S.wstride] == p) ? 1u : 0u;
                uint32_t w[4];
                philox(P, E.env_id, E.episode, ctr2(SITE_DESP, E.turn, rank >> 2), p, w);
                if ((uint64_t)pick4(w, rank & 3u) >= P.thr_keep) keepmask |= 1ull << k;
            }
            group_sync(coop);                       // every lane of the group has read the slots
            if (group_leader(coop)) {
                WAB_ROLLED
                for (uint32_t k = 0; k < E.nw; ++k)
                    if ((keepmask >> k) & 1ull) {
                        S.wolves[(int32_t)kept * S.wstride] = S.wolves[(int32_t)k * S.wstride];
                        ++kept;
                    }
            }
            group_sync(coop);
            E.nw = popc32((uint32_t)keepmask) + popc32((uint32_t)(keepmask >> 32));
        }
    }
    WAB_PC_MARK(PC_DESPAWN);

    // ---- :266 the frame the rest of the step reads: bushes with food > 0, ostrich status
    O.bm[0] = E.m[0]; O.bm[1] = E.m[1]; O.bm[2] = E.m[2]; O.bm[3] = E.m[3];
    const uint32_t status_pre = E.status;

    // ---- :267-297 wolves chase (ties -> x axis), kill on contact; wolf plane after the move (:289)
    O.wm[0] = O.wm[1] = O.wm[2] = O.wm[3] = 0u;
    if (any_wolf) {
        WAB_ROLLED
        for (uint32_t k = 0; k < E.nw; ++k) {
            const uint32_t p = S.wolves[(int32_t)k * S.wstride];
            int32_t wx = unpack_x(p), wy = unpack_y(p);
            int32_t ddx = E.x - wx, ddy = E.y - wy;                                  // :59-60
            if (P.wolves_can_move) {
                const int32_t ax = ddx < 0 ? -ddx : ddx, ay = ddy < 0 ? -ddy : ddy;
                const int32_t sx = (ddx > 0) - (ddx < 0), sy = (ddy > 0) - (ddy < 0);
                wx += (ax >= ay) ? sx : 0;                                           // :278-280
                wy += (ax < ay) ? sy : 0;                                            // :281-283
                group_sync(coop);                                                    // all lanes hold the old position
                if (group_leader(coop)) S.wolves[(int32_t)k * S.wstride] = pack_xy(wx, wy);   // :285-286
                ddx = E.x - wx; ddy = E.y - wy;
            }
            if (ddx == 0 && ddy == 0 && !P.god_mode) E.status = 2u;                  // :292-297
            if (ddx >= -HALF && ddx <= HALF && ddy >= -HALF && ddy <= HALF)          // :416-427
                setbit128(O.wm, 11 * (ddx + HALF) + (ddy + HALF), 1u);
        }
        if (E.nw && P.wolves_can_move) group_sync(coop);                             // moved positions published to the group
    }
    WAB_PC_MARK(PC_CHASE);

    // ---- :300-313 eat (bush and status as of the frame above; role is fresh)
    O.ate = 0;
    E.stale = 0u;
    const bool eat = active && ((O.bm[1] >> 28) & 1u) && (E.role == 1u || P.lookout_only) && status_pre == 0u;   // bit 60 = [5][5]
    if (WAB_ANY(eat)) {
        WAB_PC_COUNT(PP_EAT);
        if (eat) {
            O.ate = 1u;
            if (F64) {
                double f = E.food_f + P.food_inc;                                    // :307-309
                f = f < 0.0 ? 0.0 : f; f = f > 1.0 ? 1.0 : f;                        // :310
                E.food_f = f;
            } else {
                int32_t f = E.food_i + P.food_int_inc;
                E.food_i = f > P.food_int_max ? P.food_int_max : f;
            }
            // bush.food -= 1 (:312): count the eat; the cell disappears when eats == its first-reveal value
            const uint32_t cell = pack_xy(E.x, E.y);
            int32_t l = log_find(E, S, cell);
            uint32_t eats;
            if (l >= 0) {
                WAB_PC_COUNT(PP_EAT_HIT);
                eats = (uint32_t)S.logcnt[(int64_t)l * S.lstride] + 1u;
                group_sync(coop);                      // every lane of the group has read the old count
                if (group_leader(coop)) S.logcnt[(int64_t)l * S.lstride] = (uint8_t)eats;
                group_sync(coop);
            } else if (E.nlog < (uint32_t)P.log_cap) {
                eats = 1u;
                S.logcell[(int64_t)E.nlog * S.lstride] = cell;
                S.logcnt[(int64_t)E.nlog * S.lstride] = 1;
                E.nlog += 1;
                E.logsig |= cell_sig(cell);
            } else {
                eats = 1u; O.overflow = 1u;            // counted, never silent (WAB_STAT_OVERFLOWS)
            }
            const uint32_t still = eaten_bush_alive(P, E, E.x, E.y, eats);
            if (!still) { E.m[1] &= ~(1u << 28); E.dep = 1u; E.stale = 1u; }
        }
    }
    WAB_PC_MARK(PC_EAT);

    // ---- :316-322 hunger, starvation (overrides killed)
    if (F64) {
        const double f = E.food_f - P.food_dec;
        E.status = f <= 0.0 ? 1u : E.status;
        E.food_f = f <= 0.0 ? 0.0 : f;
    } else {
        const int32_t f = E.food_i - 1;
        E.status = f <= 0 ? 1u : E.status;
        E.food_i = f <= 0 ? 0 : f;
    }

    // ---- :325-326 spawn_wolves on the 48 ring cells around the moved ostrich: one binomial-first draw
    const bool spawn = P.wolves && active && D.spawn >= P.spawn_cdf[0];   // rare (2.4 % of steps): at least one wolf appears
    if (WAB_ANY(spawn)) {
        WAB_PC_COUNT(PP_SPAWN);
        if (spawn) {
            uint32_t chosen[4];
            binomial_choose(P, E.env_id, E.episode, SITE_SPAWN, E.turn, RING, D.spawn, chosen);
            WAB_ROLLED
            for (int w = 0; w < 2; ++w) {                                         // :571-574, ring order
                uint32_t bits = w ? chosen[1] : chosen[0];
                WAB_ROLLED
                while (bits) {
#if defined(__CUDA_ARCH__)
                    const int j = 32 * w + __ffs((int)bits) - 1;
#else
                    const int j = 32 * w + __builtin_ctz(bits);
#endif
                    bits &= bits - 1u;
                    int32_t ox, oy;
                    ring_offset(j, ox, oy);
                    if (E.nw < (uint32_t)P.wolf_cap) {
                        S.wolves[(int32_t)E.nw * S.wstride] = pack_xy(E.x + ox, E.y + oy);
                        E.nw += 1;
                    } else {
                        O.overflow = 1u;
                    }
                }
            }
        }
    }
    // ---- :328-340 reward, done
    const uint32_t outcome = E.status == 0u ? ((E.turn >= (uint32_t)P.max_turns) ? 1u : 0u) : (E.status == 1u ? 2u : 3u);
    O.outcome = outcome;
    O.done = outcome != 0u;
    O.reward = P.reward_table[O.ate * 4u + outcome];
    O.info = outcome | (O.ate << 2) | (O.bad_action << 3) | (E.status << 4);

    // ---- :342, :387-391, :450-452 scalar observation (fresh)
    O.food_obs = food_observation(P, E, F64);
    O.role = E.role;
    O.status = E.status;
    WAB_PC_MARK(PC_TAIL);
}

// ------------------------------------------------------------------ reset pieces (wab_env.py:231-248)
// The 36 bush blocks and 31 wolf-init groups of a reset are independent Philox calls; the kernels
// fan them out over the lanes of a warp. These two helpers are one lane's share.

// bush block blk (0..35) of the reset window -> occupancy bits (generate_bushes at reset, :244).
// The block's four cells are bits base, base+1, base+11, base+12 of the window (base = the cell with
// the larger x and y), so they are deposited as one 13-bit pattern.
WAB_HD void reset_bush_block(const Params& P, uint32_t ka, uint32_t kb, int blk, uint32_t part[4]) {
    const int32_t xb = blk / 6 - 3, yb = blk % 6 - 3;       // x >> 1 for x in [-5, 5] is [-3, 2]
    uint32_t p[2];
    const uint32_t c0 = pack_xy(xb, yb) ^ ka;
    philox2(P, c0, kb, p);
    // half-word lane = (x&1) | (y&1)<<1 : word (y&1), upper half iff (x&1)
    uint32_t h[4] = {p[0] & 0xFFFFu, p[0] >> 16, p[1] & 0xFFFFu, p[1] >> 16};
    const uint32_t t_hi = P.thr_bush1 >> 16;
    uint32_t on[4];
    on[0] = h[0] > t_hi; on[1] = h[1] > t_hi; on[2] = h[2] > t_hi; on[3] = h[3] > t_hi;
    if (h[0] == t_hi || h[1] == t_hi || h[2] == t_hi || h[3] == t_hi) {      // tie: full 32-bit draws decide
        WAB_ROLLED
        for (uint32_t l = 0; l < 4u; ++l) {
            const uint32_t v = bush_word_rare(c0, kb, P.rk2[0], l) >= P.thr_bush1 ? 1u : 0u;
            if (l == 0u) on[0] = v; else if (l == 1u) on[1] = v; else if (l == 2u) on[2] = v; else on[3] = v;
        }
    }
    const bool has = P.n_bush_thr > 0;
    const bool x0 = xb > -3, y0 = yb > -3;                   // x = 2*xb (resp. y = 2*yb) is -6 when xb = -3: outside
    // [i][j] = [5 - x][5 - y]
    const uint32_t b11 = has ? on[3] : 0u;                   // x = 2xb+1, y = 2yb+1 -> base
    const uint32_t b10 = (has && y0) ? on[1] : 0u;           // x = 2xb+1, y = 2yb   -> base + 1
    const uint32_t b01 = (has && x0) ? on[2] : 0u;           // x = 2xb,   y = 2yb+1 -> base + 11
    const uint32_t b00 = (has && x0 && y0) ? on[0] : 0u;     // x = 2xb,   y = 2yb   -> base + 12
    const uint32_t pat = b11 | (b10 << 1) | (b01 << 11) | (b00 << 12);
    const int base = 11 * (4 - 2 * xb) + (4 - 2 * yb);       // 0 .. 120
    const uint32_t r = (uint32_t)base & 31u;
    const int q = base >> 5;
    const uint32_t lo = pat << r, hi = fshl(pat, 0u, r);     // hi = pat >> (32 - r), 0 when r = 0
    part[0] |= (q == 0) ? lo : 0u;
    part[1] |= (q == 1) ? lo : ((q == 0) ? hi : 0u);
    part[2] |= (q == 2) ? lo : ((q == 1) ? hi : 0u);
    part[3] |= (q == 3) ? lo : ((q == 2) ? hi : 0u);
}
// initialize_wolves (:578-593): one binomial-first draw over the 121 window cells, c = (x+5)*11 + (y+5).
// Appends the wolves of a freshly reset env (executed by the lanes that own the env).
WAB_HD void reset_init_wolves(const Params& P, Env& E, const Slots& S, uint32_t& overflow) {
    const uint64_t v = binomial_draw(P, E.env_id, E.episode, SITE_INIT, 0u);
    if (v < P.init_cdf[0]) return;                     // 94 % of resets start without a wolf in view
    uint32_t chosen[4];
    binomial_choose(P, E.env_id, E.episode, SITE_INIT, 0u, CELLS, v, chosen);
    WAB_ROLLED
    for (int w = 0; w < 4; ++w) {
        uint32_t bits = w == 0 ? chosen[0] : w == 1 ? chosen[1] : w == 2 ? chosen[2] : chosen[3];
        WAB_ROLLED
        while (bits) {
#if defined(__CUDA_ARCH__)
            const int c = 32 * w + __ffs((int)bits) - 1;
#else
            const int c = 32 * w + __builtin_ctz(bits);
#endif
            bits &= bits - 1u;
            if (E.nw < (uint32_t)P.wolf_cap) {
                S.wolves[(int32_t)E.nw * S.wstride] = pack_xy(c / 11 - HALF, c % 11 - HALF);
                E.nw += 1;
            } else {
                overflow = 1u;
            }
        }
    }
}
// scalar part of a reset: spawn_ostriches (:595-611)
template <bool F64>
WAB_HD void reset_scalars(const Params& P, Env& E) {
    E.episode += 1;                 // first reset -> episode 0 (state is created with 0xFFFFFFFF)
    E.turn = 0; E.x = 0; E.y = 0; E.status = 0; E.nw = 0; E.nlog = 0; E.dep = 0; E.stale = 0; E.logsig = 0;
    E.role = (uint32_t)(P.starting_role < 0 ? 0 : P.starting_role);
    E.food_i = P.food_int_start;
    E.food_f = P.food_start;
    uint32_t w[4];
    philox(P, E.env_id, E.episode, ctr2(SITE_START, 0, 0), 0u, w);
    E.bk_a = w[2]; E.bk_b = w[3];                                         // bush key of the new episode
    if (P.starting_role < 0) E.role = w[1] >> 31;                         // np.random.randint(2), :598-599
    if (P.food_random) E.food_f = (double)w[0] * (1.0 / 4294967296.0);    // np.random.random(), :596-597
    (void)F64;
}

// 363-bit observation string of one env as 11 words (bits 0..120 wolves, 121..241 bushes,
// 242..362 ostriches; bit 302 = ostrich [5][5], never masked). wm / bm are the planes as observed
// (mask_grid, wab_env.py:344-357, already applied by apply_view_mask).
WAB_HD void compose_obs(const uint32_t wm[4], const uint32_t bm[4], uint32_t B[11]) {
    B[0] = wm[0]; B[1] = wm[1]; B[2] = wm[2];
    B[3] = wm[3] | (bm[0] << 25);                  // 121 = 3*32 + 25
    B[4] = (bm[0] >> 7) | (bm[1] << 25);
    B[5] = (bm[1] >> 7) | (bm[2] << 25);
    B[6] = (bm[2] >> 7) | (bm[3] << 25);
    B[7] = bm[3] >> 7;
    B[8] = 0u;
    B[9] = 1u << 14;                               // 242 + 60 = 302 = 9*32 + 14
    B[10] = 0u;
}

WAB_HD void apply_view_mask(const Params& P, uint32_t role, uint32_t wm[4], uint32_t bm[4]) {   // mask_grid :344-357
    if (!P.restrict_view) return;
    for (int w = 0; w < 4; ++w) {
        const uint32_t blind = role == 1u ? P.mask_gath[w] : P.mask_look[w];
        wm[w] &= ~blind; bm[w] &= ~blind;
    }
}

}  // namespace wab
