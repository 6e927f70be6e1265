// wab_kernels.cu — sm_100a kernels + the C ABI of include/wab_b200.h.
//
// Execution model (B200: 148 SMs, HBM-bound byte/integer work, no tensor cores on this path):
//   * one THREAD per environment runs the scalar game rules of wab_core.cuh with its state in
//     registers (struct-of-arrays in HBM, one coalesced load/store per field per launch — in the
//     multi-step kernel the state never leaves registers between steps);
//   * one WARP cooperates on the two pieces that are wide: (a) a reset fans its 36 + 31 independent
//     Philox calls over the 32 lanes and OR-reduces the window with redux.sync; (b) the observation:
//     each lane writes its env's 363-bit string into a shared-memory bit stream whose bit b is
//     exactly byte b of the warp's contiguous 32 x [3][11][11] u8 output, then the warp expands the
//     stream 16 bits -> 16 bytes per lane and issues fully coalesced 16-byte streaming stores.
//   * per-(env, episode, turn, cell) Philox4x32-10 counters make every draw order-free
//     (oracle/keyed_rng.py states the contract).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cmath>
#include <new>
#include <string>
#include <type_traits>

#include "../../include/wab_b200.h"
#include "wab_core.cuh"
#include "wab_features.cuh"
#include "wab2_core.cuh"
#include "wab_params.h"

using namespace wab;

#ifndef WAB_FLUSH_UNROLL
#define WAB_FLUSH_UNROLL 2
#endif

namespace {

constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int kFlushUnroll = WAB_FLUSH_UNROLL;
#ifndef WAB_THREADS_LPEN
#define WAB_THREADS_LPEN 64
#endif
#ifndef WAB_MIN_BLOCKS_LPEN
#define WAB_MIN_BLOCKS_LPEN 1         // lanes-per-env kernels: no register cap (one wave of few CTAs anyway)
#endif
#ifndef WAB_PIPE_PAIRS
#define WAB_PIPE_PAIRS 4              // rule/publisher warp pairs per CTA of the pipelined multi-step kernel
#endif
#ifndef WAB_THREADS_LPE1
#define WAB_THREADS_LPE1 32           // thread-per-env kernel: one warp per CTA (no intra-CTA imbalance over a T-step launch:
                                      // 1.32e10 vs 1.29e10 env-steps/s at 1M envs with 128-thread CTAs, profiles/r1f_wave_quantization.txt)
#endif
#ifndef WAB_MIN_BLOCKS_LPE1
#define WAB_MIN_BLOCKS_LPE1 (768 / WAB_THREADS_LPE1)   // cap registers at 80 so 24 warps (6 CTAs of 128) fit an SM
#endif
// h->mb counts resident CTAs per SM in units of 128 threads (6, 7, 8 = 24, 28, 32 warps)
constexpr int kMbScale = 128 / WAB_THREADS_LPE1;

struct StatePtrs {
    uint32_t* pos;       // [N]  x:i16 | y:i16 << 16
    uint32_t* misc;      // [N]  food_i:8 | role:1 | status:2 | nw (low 4 bits):4 | depleted:1 | turn:16
    uint32_t* episode;   // [N]
    uint4* bush;         // [N]  121-bit window occupancy
    uint16_t* nlog;      // [N]  entries in the depletion log : 8 | stale centre bush : 1 | nw (high 3 bits) : 3
    uint32_t* logsig;    // [N]  Bloom signature of the depletion log
    uint2* bkey;         // [N]  the episode's bush key
    double* food;        // [N]  F64 mode only
    uint32_t* wolves;    // [wolf_cap][N]
    uint32_t* logcell;   // [log_cap][N]
    uint8_t* logcnt;     // [log_cap][N]
    unsigned long long* stats;  // [8]  totals, refreshed by wab_stats_reduce_kernel when somebody asks
    unsigned long long* wstats; // [warps of the grid][8]  every warp accumulates into its own row: no atomics, no barrier
    uint32_t* hist;      // [hist_len][N] ostrich position after turn t of the current episode, or null (egocentric observations only)
    int32_t hist_len;
    int64_t n;
};

struct OutPtrs {
    uint8_t* grids; uint8_t* food; uint8_t* role; uint8_t* status;
    float* reward; uint8_t* done; uint8_t* info;
    uint8_t* features;   // optional [..][28] PragmaticObsWrapper features (wab_features.cuh)
};

template <bool F64>
__device__ __forceinline__ void load_env(const Params& P, const StatePtrs& st, int64_t idx, Env& E,
                                         uint32_t* wolves_s, int wstride) {
    const uint32_t pos = st.pos[idx], misc = st.misc[idx];
    E.x = unpack_x(pos); E.y = unpack_y(pos);
    E.food_i = (int32_t)(misc & 0xFFu);
    E.role = (misc >> 8) & 1u; E.status = (misc >> 9) & 3u; E.nw = (misc >> 11) & 15u; E.dep = (misc >> 15) & 1u;
    E.turn = misc >> 16;
    E.episode = st.episode[idx];
    const uint4 b = st.bush[idx];
    E.m[0] = b.x; E.m[1] = b.y; E.m[2] = b.z; E.m[3] = b.w;
    { const uint32_t nl = st.nlog[idx]; E.nlog = nl & 0xFFu; E.stale = (nl >> 8) & 1u; E.nw |= ((nl >> 9) & 7u) << 4; }
    E.logsig = st.logsig[idx];
    { const uint2 bk = st.bkey[idx]; E.bk_a = bk.x; E.bk_b = bk.y; }
    E.food_f = F64 ? st.food[idx] : 0.0;
    E.env_id = (uint32_t)global_env_id(P, idx);
    WAB_ROLLED
    for (uint32_t k = 0; k < E.nw; ++k) wolves_s[k * wstride] = st.wolves[(int64_t)k * st.n + idx];
}

template <bool F64>
__device__ __forceinline__ void store_env(const StatePtrs& st, int64_t idx, const Env& E,
                                          const uint32_t* wolves_s, int wstride) {
    st.pos[idx] = pack_xy(E.x, E.y);
    st.misc[idx] = ((uint32_t)E.food_i & 0xFFu) | (E.role << 8) | (E.status << 9) | ((E.nw & 15u) << 11) | (E.dep << 15) |
                   (E.turn << 16);
    st.episode[idx] = E.episode;
    st.bush[idx] = make_uint4(E.m[0], E.m[1], E.m[2], E.m[3]);
    st.nlog[idx] = (uint16_t)(E.nlog | (E.stale << 8) | ((E.nw >> 4) << 9));
    st.logsig[idx] = E.logsig;
    st.bkey[idx] = make_uint2(E.bk_a, E.bk_b);
    if (F64) st.food[idx] = E.food_f;
    WAB_ROLLED
    for (uint32_t k = 0; k < E.nw; ++k) st.wolves[(int64_t)k * st.n + idx] = wolves_s[k * wstride];
}

// Reset every env of the warp whose `need` is set (wab_env.py:231-248). All 32 lanes must call; the
// 36 bush-block Philox calls of ONE reset are spread over the 32 lanes whatever
// LPE is. `need` is replicated over the LPE lanes of a group. On return the lanes of a reset env
// hold the fresh state and its observation planes.
template <bool F64, int LPE>
__device__ __forceinline__ void warp_reset(const Params& P, Env& E, const Slots& S, bool need, int lane,
                                           uint32_t wm[4], uint32_t bm[4], uint32_t& overflow) {
    unsigned todo = __ballot_sync(FULL, need);
    if (need) reset_scalars<F64>(P, E);
    while (todo) {
        const int r = __ffs((int)todo) - 1;                       // first lane of the group to reset
        todo &= (LPE == 32) ? 0u : ~(((1u << (LPE & 31)) - 1u) << r);
        const bool mine = (lane / LPE) == (r / LPE);
        const uint32_t ka = __shfl_sync(FULL, E.bk_a, r);
        const uint32_t kb = __shfl_sync(FULL, E.bk_b, r);
        uint32_t part[4] = {0u, 0u, 0u, 0u};
#pragma unroll 1
        for (int blk = lane; blk < 36; blk += 32) reset_bush_block(P, ka, kb, blk, part);    // 36 blocks over 32 lanes
        const uint32_t m0 = __reduce_or_sync(FULL, part[0]);
        const uint32_t m1 = __reduce_or_sync(FULL, part[1]);
        const uint32_t m2 = __reduce_or_sync(FULL, part[2]);
        const uint32_t m3 = __reduce_or_sync(FULL, part[3]);
        if (mine) { E.m[0] = m0; E.m[1] = m1; E.m[2] = m2; E.m[3] = m3; }
    }
    if (need && P.wolves) reset_init_wolves(P, E, S, overflow);       // one Philox call per reset env
    if (need) {
        wolf_plane(E, S, wm);
        bm[0] = E.m[0]; bm[1] = E.m[1]; bm[2] = E.m[2]; bm[3] = E.m[3];
    }
}

__device__ __forceinline__ uint32_t nibble_to_bytes(uint32_t n) { return (n * 0x00204081u) & 0x01010101u; }

// Observation output of one WARP for one step.
//
// The warp's EPW envs own the contiguous byte range [b0, b0 + 363*EPW) of the grids tensor. Their
// 363-bit strings are concatenated into a shared-memory bit stream in which bit (off + k) is byte
// (b0 + k) of the output, off = b0 & 15 — so the stream is aligned to the 16-byte store grid whatever
// b0 is. Each lane then expands 16 bits into 16 bytes ((nibble * 0x00204081) & 0x01010101) and issues
// one coalesced 16-byte streaming store; the < 16 ragged bytes at either end, which share a store
// slot with the neighbouring warp, are written as single bytes. No CTA barrier, no atomics: the last
// 60 bits of every env's string are zero, so a word shared by two envs is written by the later one.
template <int EPW>
struct WarpStream {
    static constexpr int WORDS = (EPW * OBS_BYTES + 31 + 31) / 32 + 1;   // the slab may start at any of 32 bit offsets
};

__device__ __forceinline__ void stream_put(uint32_t* stream, int bit0, bool last, int total_bits,
                                           const uint32_t wm[4], const uint32_t bm[4], bool active) {
    uint32_t B[11];
    if (active) {
        compose_obs(wm, bm, B);
    } else {
#pragma unroll
        for (int k = 0; k < 11; ++k) B[k] = 0u;
    }
    const uint32_t sh = (uint32_t)bit0 & 31u;
    const int fw = bit0 >> 5;
    // words this env must write: up to (not including) the next env's first word; the last env also
    // zero-fills the tail of the stream so no stale shared memory is ever flushed
    const int nown = (last ? ((total_bits + 31) >> 5) : ((bit0 + OBS_BYTES) >> 5)) - fw;   // 11, 12 or 13
    stream[fw] = B[0] << sh;
#pragma unroll
    for (int k = 1; k < 11; ++k) stream[fw + k] = fshl(B[k - 1], B[k], sh);
    if (nown > 11) stream[fw + 11] = fshl(B[10], 0u, sh);
    if (nown > 12) stream[fw + 12] = 0u;
}

constexpr int kObsAlign = 16;     // the store grid the warp's bit stream is aligned to
// byte offset of an output address inside its store-grid cell (the address minus this is kObsAlign-aligned)
__device__ __forceinline__ int obs_align_off(const uint8_t* p) { return (int)(reinterpret_cast<uintptr_t>(p) & (uintptr_t)(kObsAlign - 1)); }

// gA = kObsAlign-aligned address of stream bit 0; valid bits are [off, end).
// `lut` = 256 x uint2 in shared memory: byte value -> its 8 bits as 8 bytes (built once per CTA).
// USE_LUT = false expands with two multiplies per 8 bytes instead (the lanes-per-env kernels: few chunks per step, and no
// table means no CTA barrier anywhere in a single-step launch).
// `lane`: the flushing lane of the warp.
template <bool USE_LUT = true>
__device__ __forceinline__ void stream_flush(const uint32_t* stream, const uint2* lut, uint8_t* gA, int off, int end,
                                             int lane, bool lut_built = true) {
    constexpr int SH = 4, CH = 1 << SH;                          // chunk = one 16-byte store
    const int c_lo = (off + CH - 1) >> SH, c_hi = end >> SH;     // chunks entirely inside [off, end)
    const uint16_t* hs = reinterpret_cast<const uint16_t*>(stream);
#pragma unroll kFlushUnroll
    for (int c = c_lo + lane; c < c_hi; c += 32) {
        const uint32_t h = hs[c];
        uint2 lo, hi;
        if (USE_LUT && lut_built) {
            lo = lut[h & 0xFFu]; hi = lut[h >> 8];
        } else {
            lo = make_uint2(nibble_to_bytes(h & 15u), nibble_to_bytes((h >> 4) & 15u));
            hi = make_uint2(nibble_to_bytes((h >> 8) & 15u), nibble_to_bytes(h >> 12));
        }
        __stcs(reinterpret_cast<uint4*>(gA) + c, make_uint4(lo.x, lo.y, hi.x, hi.y));
    }
    if (lane < CH) {                                              // ragged head and tail, one byte per lane
        const int head_end = min(c_lo << SH, end);
        const int hb = off + lane;
        if (hb < head_end) gA[hb] = (uint8_t)((stream[hb >> 5] >> (hb & 31)) & 1u);
        const int tb = max(c_hi << SH, head_end) + lane;
        if (tb < end) gA[tb] = (uint8_t)((stream[tb >> 5] >> (tb & 31)) & 1u);
    }
}

__device__ __forceinline__ void write_scalars(const OutPtrs& out, int64_t o, const StepOut& O) {
    out.food[o] = (uint8_t)O.food_obs;
    out.role[o] = (uint8_t)O.role;
    out.status[o] = (uint8_t)O.status;
    if (out.reward) out.reward[o] = O.reward;
    if (out.done) out.done[o] = (uint8_t)O.done;
    if (out.info) out.info[o] = (uint8_t)O.info;
}

// PragmaticObsWrapper features of the observation just produced: 28 bytes = 7 words per env
__device__ __forceinline__ void write_features(uint8_t* features, int64_t o, const StepOut& O) {
    uint32_t f[7];
    pragmatic_features(O.wm, O.bm, O.food_obs, O.role, O.status, f);
    uint32_t* dst = reinterpret_cast<uint32_t*>(features + o * FEAT_BYTES);
#pragma unroll
    for (int k = 0; k < 7; ++k) dst[k] = f[k];
}

__device__ __forceinline__ void flush_stats_row(unsigned long long* wstats, int64_t row, const uint32_t c[8]) {
    // warp redux, then lane k adds total k to the warp's own row (one 64-byte read-modify-write, exclusive to this warp)
    const int lane = threadIdx.x & 31;
    uint32_t mine = 0u;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint32_t s = __reduce_add_sync(FULL, c[k]);
        mine = lane == k ? s : mine;
    }
    if (lane < 8 && mine) wstats[row * 8 + lane] += (unsigned long long)mine;
}
__device__ __forceinline__ void flush_stats(unsigned long long* wstats, const uint32_t c[8]) {
    flush_stats_row(wstats, ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, c);
}

// totals[k] = sum over warps of wstats[warp][k]; one block per counter
__global__ void wab_stats_reduce_kernel(const unsigned long long* __restrict__ wstats, int64_t n_warps,
                                        unsigned long long* __restrict__ totals) {
    __shared__ unsigned long long part[256];
    const int k = blockIdx.x;
    unsigned long long acc = 0ull;
    for (int64_t w = threadIdx.x; w < n_warps; w += blockDim.x) acc += wstats[w * 8 + k];
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int s2 = 128; s2 > 0; s2 >>= 1) {
        if ((int)threadIdx.x < s2) part[threadIdx.x] += part[threadIdx.x + s2];
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[k] = part[0];
}

// Programmatic dependent launch (sm_90+): consecutive launches of a stream or graph overlap the next launch's
// scheduling and prologue with this launch's tail. A no-op when the launch carries no programmatic dependency.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void build_lut(uint2* lut) {
    for (int b = threadIdx.x; b < 256; b += blockDim.x)
        lut[b] = make_uint2(nibble_to_bytes((uint32_t)b & 15u), nibble_to_bytes((uint32_t)b >> 4));
    __syncthreads();
}

// Geometry: a warp owns EPW = 32 / LPE envs. Thread-per-env uses 128-thread CTAs; the lanes-per-env variants
// serve small batches where the grid is about one wave, so they use 64-thread CTAs to spread evenly over 148 SMs.
template <int LPE> struct Geo {
    static constexpr int THREADS = LPE == 1 ? WAB_THREADS_LPE1 : WAB_THREADS_LPEN;
    static constexpr int EPW = 32 / LPE;
    static constexpr int EPB = THREADS / LPE;
    static constexpr int STREAM = ((THREADS / 32) * WarpStream<EPW>::WORDS + 1) & ~1;   // even: keeps the LUT 8-byte aligned
    static constexpr int MIN_BLOCKS = LPE == 1 ? WAB_MIN_BLOCKS_LPE1 : WAB_MIN_BLOCKS_LPEN;
};

struct Ctx {   // per-thread view of the geometry
    int lane, sub, slot;          // slot = env index within the warp
    int env_local;                // env index within the CTA
    int64_t idx, warp_first;      // global env index; first env of the warp
    int n_valid;                  // envs of the warp that exist
    bool active, writer;          // env exists; this lane writes the env's outputs
};

template <int LPE>
__device__ __forceinline__ Ctx make_ctx(int64_t n) {
    Ctx c;
    constexpr int EPB = Geo<LPE>::EPB, EPW = Geo<LPE>::EPW;
    c.lane = threadIdx.x & 31;
    c.sub = LPE == 1 ? 0 : (c.lane % LPE);
    c.slot = c.lane / LPE;
    c.env_local = threadIdx.x / LPE;
    c.idx = (int64_t)blockIdx.x * EPB + c.env_local;
    c.warp_first = c.idx - c.slot;
    c.active = c.idx < n;
    c.writer = c.active && c.sub == 0;
    const int64_t left = n - c.warp_first;
    c.n_valid = (int)(left < EPW ? (left > 0 ? left : 0) : EPW);
    return c;
}

// Publish the warp's observations for one step; `first_byte` = byte offset of the warp's first env
// in the grids tensor (any alignment).
template <int LPE>
__device__ __forceinline__ void emit_obs(uint32_t* stream, const uint2* lut, const Ctx& c, uint8_t* grids,
                                         int64_t first_byte, const uint32_t wm[4], const uint32_t bm[4], bool lut_built = true) {
    constexpr int EPW = Geo<LPE>::EPW;
    const int off = obs_align_off(grids + first_byte);
    const int total = off + EPW * OBS_BYTES;
    if (c.sub == 0)
        stream_put(stream, off + OBS_BYTES * c.slot, c.slot == EPW - 1, total, wm, bm, c.active);
    __syncwarp();
    stream_flush<true>(stream, lut, grids + (first_byte - off), off, off + OBS_BYTES * c.n_valid, c.lane, lut_built);
    __syncwarp();
}

// T lockstep steps of every env; observation, reward, done and info are written for every step.
// MB = resident CTAs per SM the register budget is capped for (the thread-per-env kernel also exists for 7 and 8,
// picked at create when that makes a batch fit in ONE wave: 131,072 envs are 1.15 waves of 6 CTAs per SM).
template <bool F64, int LPE, int MB = Geo<LPE>::MIN_BLOCKS>
__global__ void __launch_bounds__(Geo<LPE>::THREADS, MB)
wab_step_kernel(const __grid_constant__ Params P, const StatePtrs st, const uint8_t* __restrict__ actions,
                const int n_steps, const OutPtrs out) {
    extern __shared__ uint32_t smem[];
    constexpr int EPB = Geo<LPE>::EPB;
    const int64_t n = st.n;
    const Ctx c = make_ctx<LPE>(n);
    uint32_t* wolves_s = smem + c.env_local;                                  // [wolf_cap][EPB]
    uint32_t* stream = smem + P.wolf_cap * EPB + (threadIdx.x >> 5) * WarpStream<Geo<LPE>::EPW>::WORDS;
    uint2* lut = reinterpret_cast<uint2*>(smem + P.wolf_cap * EPB + Geo<LPE>::STREAM);   // 256 x 8 bytes (thread-per-env only)
    // The 256-entry byte-expansion table (and the CTA barrier that publishes it) serves the thread-per-env kernel, whose
    // ALU pipes are the bottleneck; the lanes-per-env kernels expand with multiplies: measured on one box at 4,096 envs,
    // 240 steps per launch, 1.757e9 env-steps/s without the table against 1.703e9 with it (profiles/r2_ab_small_batch.txt).
    const bool lut_built = LPE == 1;
    pdl_launch_dependents();               // the next launch may be scheduled now; it waits below before touching state
    if (lut_built) build_lut(lut);
    pdl_wait();                            // everything this launch reads or writes follows the previous launch
    Coop<LPE> coop;
    coop.sub = (uint32_t)c.sub;
    coop.gmask = LPE == 32 ? FULL : (((1u << (LPE & 31)) - 1u) << (c.lane - c.sub));

    Env E;
    Slots S;
    S.wolves = wolves_s; S.wstride = EPB;
    S.logcell = st.logcell + (c.active ? c.idx : 0); S.logcnt = st.logcnt + (c.active ? c.idx : 0); S.lstride = n;
    if (c.active) load_env<F64>(P, st, c.idx, E, wolves_s, EPB);
    else { E = Env(); }

    // statistics as packed 16-bit fields (n_steps <= 65535): one 64-bit add per step instead of seven
    unsigned long long acc_outcome = 0ull;   // [alive, finished, starved, killed] counts
    unsigned long long acc_misc = 0ull;      // [eats, bad actions, overflows]
    const uint8_t* ap = actions + (c.active ? c.idx : 0);
    uint32_t a_next = c.active ? *ap : 0u;
    int64_t o = c.idx;                                   // index of this env in the [T][N] outputs
    int64_t first_byte = c.warp_first * OBS_BYTES;       // byte offset of the warp's slab in the grids tensor
    for (int t = 0; t < n_steps; ++t, o += n, first_byte += n * OBS_BYTES) {
        StepOut O;
        bool need_reset = false;
        const uint32_t a = a_next;
        ap += n;
        if (c.active && t + 1 < n_steps) a_next = *ap;   // prefetch: off the critical path
        if (c.active) {
            env_step<F64, LPE>(P, E, S, a, O, coop);
            if (st.hist && c.writer && E.turn < (uint32_t)st.hist_len) st.hist[(int64_t)E.turn * n + c.idx] = pack_xy(E.x, E.y);
            need_reset = O.done && P.auto_reset;
            acc_outcome += 1ull << (16u * O.outcome);    // auto_reset = 0: every step that reports done counts
            acc_misc += (unsigned long long)O.ate | ((unsigned long long)O.bad_action << 16);
        } else {
            O = StepOut();
        }
        if (__any_sync(FULL, need_reset)) {
            warp_reset<F64, LPE>(P, E, S, need_reset, c.lane, O.wm, O.bm, O.overflow);
            if (need_reset) {          // VecEnv semantics: the post-reset observation is returned
                O.food_obs = food_observation(P, E, F64);
                O.role = E.role; O.status = E.status;
            }
        }
        apply_view_mask(P, O.role, O.wm, O.bm);            // mask_grid, wab_env.py:344-357
        if (c.writer) {
            acc_misc += (unsigned long long)O.overflow << 32;
            write_scalars(out, o, O);
            if (out.features) write_features(out.features, o, O);
        }
        if (out.grids) emit_obs<LPE>(stream, lut, c, out.grids, first_byte, O.wm, O.bm, lut_built);   // null: features-only stepping
    }
    if (c.writer) store_env<F64>(st, c.idx, E, wolves_s, EPB);
    uint32_t cnt[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    if (c.writer) {
        const uint32_t fin = (uint32_t)(acc_outcome >> 16) & 0xFFFFu, sta = (uint32_t)(acc_outcome >> 32) & 0xFFFFu,
                       kil = (uint32_t)(acc_outcome >> 48) & 0xFFFFu;
        cnt[WAB_STAT_EPISODES] = fin + sta + kil;
        cnt[WAB_STAT_STEPS] = (uint32_t)n_steps;
        cnt[WAB_STAT_FINISHED] = fin; cnt[WAB_STAT_STARVED] = sta; cnt[WAB_STAT_KILLED] = kil;
        cnt[WAB_STAT_EATS] = (uint32_t)acc_misc & 0xFFFFu;
        cnt[WAB_STAT_BAD_ACTIONS] = (uint32_t)(acc_misc >> 16) & 0xFFFFu;
        cnt[WAB_STAT_OVERFLOWS] = (uint32_t)(acc_misc >> 32) & 0xFFFFu;
    }
    flush_stats(st.wstats, cnt);
}

// ---- the multi-step kernel of the lanes-per-env geometries as a two-warp pipeline --------------------------------------
// A small batch is bound by the length of one step's dependent instruction chain, and a third of that chain is not rules
// at all: composing the 363-bit strings, expanding them to bytes, the 16-byte stores and the scalar outputs. Here a CTA is
// one PAIR of warps that owns EPW = 32 / LPE envs: warp 0 runs the rules (env_step_pipe in wab_core.cuh: wab_step_kernel's
// rules with each step's keyed draws made first and the rare paths behind warp-uniform tests) and parks
// each step's planes and scalars in a ring of shared-memory slots; warp 1 publishes them — bit stream, byte expansion,
// stores, scalars, features — while warp 0 is already on the next steps. The two meet only at mbarriers in shared memory
// (one "full" and one "empty" barrier per ring slot; an arrive never blocks, a wait spins on the barrier's phase parity).
// Results are identical to wab_step_kernel's (the same draws and rules per env); WAB_PIPE=0 selects that kernel.
template <int LPE> struct PipeGeo {
    static constexpr int EPW = 32 / LPE;
    static constexpr int DEPTH = 4;                        // ring slots, each with a full and an empty mbarrier
    static constexpr int RES = 12;                         // words parked per (env, step): 2 x 4 planes, scalars, info, reward
    static constexpr int RING = DEPTH * EPW * RES;
    static constexpr int SW = (WarpStream<EPW>::WORDS + 3) & ~3;
    // Warp w of a CTA sits on scheduler w % 4 of its SM. A CTA is therefore FOUR pairs — warps 0..3 run the rules,
    // warps 4..7 publish — so every scheduler gets the same mix of both roles; with one pair per CTA the rule warps of an
    // SM all land on two of its four schedulers and the pipeline gains nothing (profiles/r2j_pipe_ab.txt).
    static constexpr int PAIRS = WAB_PIPE_PAIRS;
    static constexpr int THREADS = 64 * PAIRS;
    static __host__ __device__ int pair_words(int wolf_cap) { return ((wolf_cap * EPW + 3) & ~3) + RING + SW + 4 * DEPTH; }
};
// Shared-memory mbarriers rather than named hardware barriers: the SM's pool of named barriers caps resident CTAs
// (2 * DEPTH + 1 of them per CTA left room for ~4 CTAs per SM; a 4,096-env batch needs 7 to be one wave).
__device__ __forceinline__ uint32_t pipe_smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void pipe_mbar_init(uint64_t* b) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pipe_smem_addr(b)), "r"(1u) : "memory");
}
// one elected lane arrives for its warp (after __syncwarp: the warp's shared-memory accesses are ordered before it; the
// arrive has release, the wait acquire semantics at CTA scope)
__device__ __forceinline__ void pipe_mbar_arrive(uint64_t* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(pipe_smem_addr(b)) : "memory");
}
__device__ __forceinline__ void pipe_mbar_wait(uint64_t* b, uint32_t parity) {
    const uint32_t a = pipe_smem_addr(b);
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}

#if defined(WAB_PIPE_CLOCKS)
// The probe's totals over every rule warp of every launch since the last wab_pipe_clocks_read(clear = 1):
// [PC_N] cycles by region, then [PP_N] passes through each rare path (PP_STEPS: warp-steps).
__device__ unsigned long long wab_pipe_clocks_buf[PC_N + PP_N];
__device__ __forceinline__ void pipe_clocks_begin() {
    const int w = (threadIdx.x >> 5) % kPcWarps;
    if ((threadIdx.x & 31) == 0) {
        for (int r = 0; r < PC_N; ++r) pc_cyc[w][r] = 0ull;
        for (int k = 0; k < PP_N; ++k) pc_cnt[w][k] = 0u;
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) pc_cyc[w][PC_N] = clock64();
}
__device__ __forceinline__ void pipe_clocks_flush() {
    __syncwarp();
    const int w = (threadIdx.x >> 5) % kPcWarps;
    if ((threadIdx.x & 31) == 0) {
        for (int r = 0; r < PC_N; ++r) atomicAdd(&wab_pipe_clocks_buf[r], pc_cyc[w][r]);
        for (int k = 0; k < PP_N; ++k) atomicAdd(&wab_pipe_clocks_buf[PC_N + k], (unsigned long long)pc_cnt[w][k]);
    }
}
#else
__device__ __forceinline__ void pipe_clocks_begin() {}
__device__ __forceinline__ void pipe_clocks_flush() {}
#endif

template <bool F64, int LPE>
__global__ void __launch_bounds__(PipeGeo<LPE>::THREADS, 1)
wab_step_pipe_kernel(const __grid_constant__ Params P, const StatePtrs st, const uint8_t* __restrict__ actions,
                     const int n_steps, const OutPtrs out) {
    extern __shared__ uint32_t smem[];
    constexpr int EPW = PipeGeo<LPE>::EPW, D = PipeGeo<LPE>::DEPTH, RES = PipeGeo<LPE>::RES;
    const int64_t n = st.n;
    const int lane = threadIdx.x & 31;
    constexpr int PAIRS = PipeGeo<LPE>::PAIRS;
    const int warp = threadIdx.x >> 5, pair = warp % PAIRS;
    const int64_t group = (int64_t)blockIdx.x * PAIRS + pair;
    const int64_t warp_first = group * EPW;
    uint32_t* pbase = smem + pair * PipeGeo<LPE>::pair_words(P.wolf_cap);
    uint32_t* ring = pbase + ((P.wolf_cap * EPW + 3) & ~3); // [DEPTH][EPW][RES], 16-byte aligned
    uint32_t* stream = ring + PipeGeo<LPE>::RING;
    uint64_t* full = reinterpret_cast<uint64_t*>(stream + PipeGeo<LPE>::SW);   // [DEPTH] step t is in slot t % DEPTH
    uint64_t* empty = full + D;                                                // [DEPTH] the slot has been read
    pdl_launch_dependents();
    if (warp >= PAIRS && lane < 2 * D) pipe_mbar_init(full + lane);
    __syncthreads();
    pdl_wait();
    if (warp < PAIRS) {
        // ---------------------------------------------------------------- warp 0: the rules
        Ctx c;
        c.lane = lane; c.sub = lane % LPE; c.slot = lane / LPE; c.env_local = c.slot;
        c.idx = warp_first + c.slot; c.warp_first = warp_first;
        c.active = c.idx < n; c.writer = c.active && c.sub == 0;
        c.n_valid = 0;
        uint32_t* wolves_s = pbase + c.env_local;          // [wolf_cap][EPW]
        Coop<LPE> coop;
        coop.sub = (uint32_t)c.sub;
        coop.gmask = LPE == 32 ? FULL : (((1u << (LPE & 31)) - 1u) << (c.lane - c.sub));
        Env E;
        Slots S;
        S.wolves = wolves_s; S.wstride = EPW;
        S.logcell = st.logcell + (c.active ? c.idx : 0); S.logcnt = st.logcnt + (c.active ? c.idx : 0); S.lstride = n;
        if (c.active) load_env<F64>(P, st, c.idx, E, wolves_s, EPW);
        else { E = Env(); }
        unsigned long long acc_outcome = 0ull, acc_misc = 0ull;
        const uint8_t* ap = actions + (c.active ? c.idx : 0);
        uint32_t a_next = c.active ? *ap : 0u;
        pipe_clocks_begin();
        for (int t = 0; t < n_steps; ++t) {
            WAB_PC_COUNT(PP_STEPS);
            StepOut O;
            const uint32_t a = a_next;
            ap += n;
            if (c.active && t + 1 < n_steps) a_next = *ap;
            env_step_pipe<F64, LPE>(P, E, S, a, O, coop, c.active);   // the whole warp, absent envs included
            if (st.hist && c.writer && E.turn < (uint32_t)st.hist_len) st.hist[(int64_t)E.turn * n + c.idx] = pack_xy(E.x, E.y);
            const bool need_reset = c.active && O.done && P.auto_reset;
            acc_outcome += c.active ? 1ull << (16u * O.outcome) : 0ull;
            acc_misc += c.active ? (unsigned long long)O.ate | ((unsigned long long)O.bad_action << 16) : 0ull;
            if (__any_sync(FULL, need_reset)) {
                WAB_PC_COUNT(PP_RESET);
                warp_reset<F64, LPE>(P, E, S, need_reset, c.lane, O.wm, O.bm, O.overflow);
                if (need_reset) {
                    O.food_obs = food_observation(P, E, F64);
                    O.role = E.role; O.status = E.status;
                }
            }
            apply_view_mask(P, O.role, O.wm, O.bm);
            WAB_PC_MARK(PC_RESET);
            const int s = t & (D - 1);
            __syncwarp();
            if (t >= D) pipe_mbar_wait(empty + s, ((uint32_t)(t / D) - 1u) & 1u);   // the publisher has taken step t - D out of this slot
            if (c.writer) {
                acc_misc += (unsigned long long)O.overflow << 32;
                uint32_t* r = ring + (s * EPW + c.slot) * RES;
                *reinterpret_cast<uint4*>(r) = make_uint4(O.wm[0], O.wm[1], O.wm[2], O.wm[3]);
                *reinterpret_cast<uint4*>(r + 4) = make_uint4(O.bm[0], O.bm[1], O.bm[2], O.bm[3]);
                *reinterpret_cast<uint4*>(r + 8) = make_uint4(O.food_obs | (O.role << 8) | (O.status << 16) | (O.done << 24),
                                                              O.info, __float_as_uint(O.reward), 0u);
            }
            __syncwarp();
            if (lane == 0) pipe_mbar_arrive(full + s);      // step t is in the slot
            WAB_PC_MARK(PC_HANDOFF);
        }
        pipe_clocks_flush();
        if (c.writer) store_env<F64>(st, c.idx, E, wolves_s, EPW);
        uint32_t cnt[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
        if (c.writer) {
            const uint32_t fin = (uint32_t)(acc_outcome >> 16) & 0xFFFFu, sta = (uint32_t)(acc_outcome >> 32) & 0xFFFFu,
                           kil = (uint32_t)(acc_outcome >> 48) & 0xFFFFu;
            cnt[WAB_STAT_EPISODES] = fin + sta + kil;
            cnt[WAB_STAT_STEPS] = (uint32_t)n_steps;
            cnt[WAB_STAT_FINISHED] = fin; cnt[WAB_STAT_STARVED] = sta; cnt[WAB_STAT_KILLED] = kil;
            cnt[WAB_STAT_EATS] = (uint32_t)acc_misc & 0xFFFFu;
            cnt[WAB_STAT_BAD_ACTIONS] = (uint32_t)(acc_misc >> 16) & 0xFFFFu;
            cnt[WAB_STAT_OVERFLOWS] = (uint32_t)(acc_misc >> 32) & 0xFFFFu;
        }
        flush_stats_row(st.wstats, group, cnt);
    } else {
        // ---------------------------------------------------------------- warp 1: the publisher (lane l < EPW: env l)
        const int64_t idx = warp_first + lane;
        const bool mine = lane < EPW && idx < n;
        const int64_t left = n - warp_first;
        const int n_valid = (int)(left < EPW ? (left > 0 ? left : 0) : EPW);
        int64_t o = idx;
        int64_t first_byte = warp_first * OBS_BYTES;
        for (int t = 0; t < n_steps; ++t, o += n, first_byte += n * OBS_BYTES) {
            const int s = t & (D - 1);
            pipe_mbar_wait(full + s, (uint32_t)(t / D) & 1u);   // step t is in the slot
            const int off = obs_align_off(out.grids + first_byte);
            uint4 sc = make_uint4(0u, 0u, 0u, 0u);
            StepOut O;
            if (lane < EPW) {
                const uint32_t* r = ring + (s * EPW + lane) * RES;
                const uint4 w = *reinterpret_cast<const uint4*>(r), b = *reinterpret_cast<const uint4*>(r + 4);
                sc = *reinterpret_cast<const uint4*>(r + 8);
                O.wm[0] = w.x; O.wm[1] = w.y; O.wm[2] = w.z; O.wm[3] = w.w;
                O.bm[0] = b.x; O.bm[1] = b.y; O.bm[2] = b.z; O.bm[3] = b.w;
                if (out.grids) stream_put(stream, off + OBS_BYTES * lane, lane == EPW - 1, off + EPW * OBS_BYTES, O.wm, O.bm, mine);
            }
            __syncwarp();                                   // every read of the slot has landed in registers or the stream
            if (lane == 0) pipe_mbar_arrive(empty + s);     // the slot is free for step t + D
            if (mine) {
                O.food_obs = sc.x & 0xFFu; O.role = (sc.x >> 8) & 0xFFu; O.status = (sc.x >> 16) & 0xFFu;
                O.done = sc.x >> 24; O.info = sc.y; O.reward = __uint_as_float(sc.z);
                write_scalars(out, o, O);
                if (out.features) write_features(out.features, o, O);
            }
            if (out.grids) stream_flush<false>(stream, nullptr, out.grids + (first_byte - off), off, off + OBS_BYTES * n_valid, lane);
            __syncwarp();
        }
    }
}

// reset(mask) + fresh observation of every env
template <bool F64, int LPE>
__global__ void __launch_bounds__(Geo<LPE>::THREADS)
wab_reset_kernel(const __grid_constant__ Params P, const StatePtrs st, const uint8_t* __restrict__ mask,
                 const OutPtrs out) {
    extern __shared__ uint32_t smem[];
    constexpr int EPB = Geo<LPE>::EPB;
    const int64_t n = st.n;
    const Ctx c = make_ctx<LPE>(n);
    uint32_t* wolves_s = smem + c.env_local;
    uint32_t* stream = smem + P.wolf_cap * EPB + (threadIdx.x >> 5) * WarpStream<Geo<LPE>::EPW>::WORDS;
    uint2* lut = reinterpret_cast<uint2*>(smem + P.wolf_cap * EPB + Geo<LPE>::STREAM);
    pdl_launch_dependents();
    if (LPE == 1) build_lut(lut);
    pdl_wait();
    const bool lut_built = LPE == 1;
    Env E;
    Slots S;
    S.wolves = wolves_s; S.wstride = EPB;
    S.logcell = st.logcell + (c.active ? c.idx : 0); S.logcnt = st.logcnt + (c.active ? c.idx : 0); S.lstride = n;
    if (c.active) load_env<F64>(P, st, c.idx, E, wolves_s, EPB);
    else { E = Env(); }
    const bool need = c.active && (mask == nullptr || mask[c.idx] != 0);
    StepOut O = StepOut();
    uint32_t cnt[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
    if (c.active && !need) {
        wolf_plane(E, S, O.wm);
        O.bm[0] = E.m[0]; O.bm[1] = E.m[1] | (E.stale << 28); O.bm[2] = E.m[2]; O.bm[3] = E.m[3];   // as last observed
    }
    warp_reset<F64, LPE>(P, E, S, need, c.lane, O.wm, O.bm, O.overflow);
    if (c.active) {
        O.food_obs = food_observation(P, E, F64);
        O.role = E.role; O.status = E.status;
    }
    apply_view_mask(P, O.role, O.wm, O.bm);
    if (c.writer) {
        out.food[c.idx] = (uint8_t)O.food_obs; out.role[c.idx] = (uint8_t)O.role; out.status[c.idx] = (uint8_t)O.status;
        if (out.features) write_features(out.features, c.idx, O);
        cnt[WAB_STAT_OVERFLOWS] += O.overflow;
        store_env<F64>(st, c.idx, E, wolves_s, EPB);
    }
    if (out.grids) emit_obs<LPE>(stream, lut, c, out.grids, c.warp_first * OBS_BYTES, O.wm, O.bm, lut_built);
    flush_stats(st.wstats, cnt);
}

// PragmaticObsWrapper.observation (wab_env.py:726-761) for an arbitrary observation batch in HBM.
__global__ void wab_features_kernel(const uint8_t* __restrict__ grids, const uint8_t* __restrict__ food,
                                    const uint8_t* __restrict__ role, const uint8_t* __restrict__ status, int64_t n,
                                    uint8_t* __restrict__ features) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    StepOut O = StepOut();
    const uint8_t* g = grids + i * OBS_BYTES;
    for (int c = 0; c < CELLS; ++c) {
        O.wm[c >> 5] |= (g[c] ? 1u : 0u) << (c & 31);
        O.bm[c >> 5] |= (g[CELLS + c] ? 1u : 0u) << (c & 31);
    }
    O.food_obs = food[i]; O.role = role[i]; O.status = status[i];
    write_features(features, i, O);
}

// gym.spaces.flatten of the wrapper's observation space (wab_env.py:710-724, actor_critic.py:188):
// one-hot of every Discrete, then the 121-cell view mask. Column k of a row whose 28 feature bytes are f.
__device__ __forceinline__ float flat_column(const Params& P, const uint8_t* f, int k, int food_dim) {
#pragma unroll
    for (int species = 0; species < 2; ++species) {
        const int base = species * 12;
        if (k < 96) return f[base + k / 12] == k % 12 ? 1.f : 0.f;                   // nearest, second: 8 x one-hot(12)
        if (k < 140) return f[base + 8 + (k - 96) / 11] == (k - 96) % 11 ? 1.f : 0.f;   // counts: 4 x one-hot(11)
        k -= 140;
    }
    if (k < 2) return f[24] == k ? 1.f : 0.f;
    if (k < 2 + food_dim) return f[25] == k - 2 ? 1.f : 0.f;
    if (k < 4 + food_dim) return f[26] == k - 2 - food_dim ? 1.f : 0.f;
    if (k < 7 + food_dim) return f[27] == k - 4 - food_dim ? 1.f : 0.f;
    const int c = k - 7 - food_dim;                                                     // view mask (obs[6])
    const uint32_t w = P.restrict_view ? (f[26] == 1 ? P.mask_gath[c >> 5] : P.mask_look[c >> 5]) : 0u;
    return (float)((w >> (c & 31)) & 1u);
}
__device__ __forceinline__ int flat_dim_of(int food_dim) { return 2 * (2 * 4 * (MAX_DISTANCE + 1) + 4 * 11) + 2 + food_dim + 2 + 3 + CELLS; }

// One thread per output element.
__global__ void wab_flatten_kernel(const __grid_constant__ Params P, const uint8_t* __restrict__ features, int64_t rows,
                                   int food_dim, float* __restrict__ outp) {
    const int dim = flat_dim_of(food_dim);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows * dim) return;
    const int64_t row = e / dim;
    outp[e] = flat_column(P, features + row * FEAT_BYTES, (int)(e - row * dim), food_dim);
}

// The policy input of actor_critic.py:188-189 in one pass: flatten + noise_scale * U[0,1) + cast. One warp per row;
// lane L owns columns L, L + 32, ... so every store instruction writes 32 consecutive elements of the row (rows are
// 449 elements long: no 16-byte alignment to exploit), the row's 28 feature bytes sit in a per-warp shared-memory slot,
// and a column is a table lookup (feature index, value) -> one compare — no division, no per-element branching (the
// first version spent 64 us on the 32,768 x 449 matrix, 7x its memory time, on 64-bit index arithmetic). One Philox
// call feeds four columns of a lane; the 64-bit draw counter lives in device memory so a captured graph gets fresh
// noise on every replay. The key is the global env id (env_id_base + row), so a shard draws what the unsharded batch
// draws for the same envs. BF16 = 0: f32 output, 1: bf16 output.
constexpr int FLAT_MAX_DIM = 2 * (2 * 4 * (MAX_DISTANCE + 1) + 4 * 11) + 2 + 256 + 2 + 3 + CELLS;
__device__ __forceinline__ uint32_t flat_descriptor(int k, int food_dim) {     // fi : 8 | value : 8 | view-mask column : 1
    for (int species = 0; species < 2; ++species) {
        const int base = species * 12;
        if (k < 96) return (uint32_t)(base + k / 12) | ((uint32_t)(k % 12) << 8);
        if (k < 140) return (uint32_t)(base + 8 + (k - 96) / 11) | ((uint32_t)((k - 96) % 11) << 8);
        k -= 140;
    }
    if (k < 2) return 24u | ((uint32_t)k << 8);
    if (k < 2 + food_dim) return 25u | ((uint32_t)(k - 2) << 8);
    if (k < 4 + food_dim) return 26u | ((uint32_t)(k - 2 - food_dim) << 8);
    if (k < 7 + food_dim) return 27u | ((uint32_t)(k - 4 - food_dim) << 8);
    return 26u | ((uint32_t)(k - 7 - food_dim) << 8) | (1u << 16);              // view mask cell, selected by the role
}
template <int BF16>
__global__ void __launch_bounds__(256) wab_flatten_noisy_kernel(const __grid_constant__ Params P, const uint8_t* __restrict__ features,
                                                                int64_t rows, int food_dim, void* __restrict__ outp, float noise_scale,
                                                                const unsigned long long* __restrict__ d_counter) {
    __shared__ uint32_t desc[FLAT_MAX_DIM];
    __shared__ uint32_t frow[8][8];                   // the 28 feature bytes of the row each warp is working on
    const int dim = flat_dim_of(food_dim);
    for (int k = threadIdx.x; k < dim; k += blockDim.x) desc[k] = flat_descriptor(k, food_dim);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long ctr = d_counter ? *d_counter : 0ull;
    const bool noisy = noise_scale != 0.f;
    const float scale = noise_scale * (1.0f / 16777216.0f);
    for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < rows; row += (int64_t)gridDim.x * 8) {
        __syncwarp();
        if (lane < 7) frow[warp][lane] = reinterpret_cast<const uint32_t*>(features + row * FEAT_BYTES)[lane];
        __syncwarp();
        const uint8_t* f = reinterpret_cast<const uint8_t*>(frow[warp]);
        const uint32_t* vm = P.restrict_view ? (f[26] == 1 ? P.mask_gath : P.mask_look) : nullptr;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        int it = 0;
        const uint64_t g = global_env_id(P, row);                  // the noise key: the row's global env id
        for (int k = lane; k < dim; k += 32, ++it) {
            if (noisy && (it & 3) == 0)
                philox(P, (uint32_t)g, (uint32_t)(g >> 32) ^ ((uint32_t)(it >> 2) << 24) ^ ((uint32_t)lane << 16), (uint32_t)ctr,
                       (uint32_t)(ctr >> 32) ^ 0x464C4154u, w);
            const uint32_t d = desc[k];
            float v;
            if (d >> 16) {
                const uint32_t c = (d >> 8) & 0xFFu;
                v = vm ? (float)((vm[c >> 5] >> (c & 31)) & 1u) : 0.f;
            } else {
                v = f[d & 0xFFu] == ((d >> 8) & 0xFFu) ? 1.f : 0.f;
            }
            if (noisy) v += scale * (float)(pick4(w, (uint32_t)it & 3u) >> 8);
            if (BF16) reinterpret_cast<__nv_bfloat16*>(outp)[row * dim + k] = __float2bfloat16_rn(v);
            else reinterpret_cast<float*>(outp)[row * dim + k] = v;
        }
    }
}

}  // namespace
#include "wab_policy_tc.cuh"
#include "wab_policy_bwd.cuh"
namespace {

// The tail of the reference's Policy.forward and select_action in one pass (actor_critic.py:84-97, :108-125): from the
// pre-activation output z3 of affine3, x = clamp(leaky_relu(z3), -4, 4); logits = action_head(x); value = value_head(x);
// probs = softmax(logits); action = Categorical(probs).sample() (inverse CDF on one keyed uniform per row) and its
// log-probability. One warp per row: each lane holds HID / 32 activations, the n_actions + 1 dot products are warp
// sums. fp32 throughout. Replaces eleven library launches (clamp, two skinny GEMMs that cuBLAS runs as 17 us gemv-style
// kernels at 32,768 rows, their bias adds, softmax, sampling, copies) with one pass over the 16 MB activation matrix.
// wab_policy_tail takes no handle, so it knows no shard: its draws are keyed by the local row.
template <int HID>
__global__ void __launch_bounds__(256) wab_policy_tail_kernel(const __grid_constant__ Params P, const float* __restrict__ z3,
                                                              const float* __restrict__ w_heads, const float* __restrict__ b_heads,
                                                              int64_t rows, int n_actions, float slope, float clamp_lo, float clamp_hi,
                                                              const unsigned long long* __restrict__ d_counter,
                                                              uint8_t* __restrict__ actions, float* __restrict__ value,
                                                              float* __restrict__ probs, float* __restrict__ logp) {
    constexpr int PER = HID / 32;
    __shared__ float wsm[9 * HID];
    const int n_out = n_actions + 1;
    for (int k = threadIdx.x; k < n_out * HID; k += blockDim.x) wsm[k] = w_heads[k];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned long long ctr = d_counter ? *d_counter : 0ull;
    for (int64_t row = (int64_t)blockIdx.x * 8 + warp; row < rows; row += (int64_t)gridDim.x * 8) {
        float x[PER];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            float v = z3[row * HID + j * 32 + lane];
            v = v > 0.f ? v : v * slope;                                  // F.leaky_relu, :92
            x[j] = fminf(fmaxf(v, clamp_lo), clamp_hi);                   // torch.clamp(x, -4, 4), :93
        }
        float acc[9];
#pragma unroll
        for (int o = 0; o < 9; ++o) {
            acc[o] = 0.f;
            if (o < n_out) {
#pragma unroll
                for (int j = 0; j < PER; ++j) acc[o] = fmaf(x[j], wsm[o * HID + j * 32 + lane], acc[o]);
#pragma unroll
                for (int sft = 16; sft > 0; sft >>= 1) acc[o] += __shfl_xor_sync(FULL, acc[o], sft);
                acc[o] += b_heads[o];
            }
        }
        float mx = -3.4e38f;
#pragma unroll
        for (int o = 0; o < 8; ++o) if (o < n_actions) mx = fmaxf(mx, acc[o]);
        float e[8], tot = 0.f;
#pragma unroll
        for (int o = 0; o < 8; ++o) { e[o] = o < n_actions ? expf(acc[o] - mx) : 0.f; tot += e[o]; }   // F.softmax, :96
        uint32_t w[4];
        philox(P, (uint32_t)(row >> 2), (uint32_t)(row >> 34), (uint32_t)ctr, (uint32_t)(ctr >> 32) ^ 0x53414D50u, w);
        const float u = (float)(pick4(w, (uint32_t)row & 3u) >> 8) * (1.0f / 16777216.0f);
        const float target = u * tot;
        float cum = 0.f, p_pick = 0.f;
        int pick = n_actions - 1;
        bool found = false;
#pragma unroll
        for (int o = 0; o < 8; ++o) {                                     // smallest a with target < e[0] + ... + e[a]
            cum += e[o];
            if (!found && o < n_actions && target < cum) { pick = o; found = true; }
        }
#pragma unroll
        for (int o = 0; o < 8; ++o) if (o == pick) p_pick = e[o];
        if (lane == 0) {
            actions[row] = (uint8_t)pick;
            if (value) value[row] = acc[n_actions < 8 ? n_actions : 8];
            if (logp) logp[row] = logf(p_pick / tot);
        }
        if (probs && lane < n_actions) {
            float mine = 0.f;
#pragma unroll
            for (int o = 0; o < 8; ++o) if (o == lane) mine = e[o];
            probs[row * n_actions + lane] = mine / tot;
        }
    }
}

// Categorical(probs).sample() of actor_critic.py:117-120 for n rows of up to 8 probabilities: inverse CDF on one keyed
// uniform per row (rows share a Philox call four at a time), keyed by the local row (wab_sample_categorical takes no
// handle, so it knows no shard). BF16 = 1: probs are bf16.
template <int BF16>
__global__ void wab_sample_kernel(const __grid_constant__ Params P, const void* __restrict__ probs, int64_t n, int n_actions,
                                  const unsigned long long* __restrict__ d_counter, uint8_t* __restrict__ actions) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long ctr = d_counter ? *d_counter : 0ull;
    uint32_t w[4];
    philox(P, (uint32_t)(i >> 2), (uint32_t)(i >> 34), (uint32_t)ctr, (uint32_t)(ctr >> 32) ^ 0x53414D50u, w);
    const float u = (float)(pick4(w, (uint32_t)i & 3u) >> 8) * (1.0f / 16777216.0f);
    float p[8], total = 0.f;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        p[a] = 0.f;
        if (a < n_actions)
            p[a] = BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(probs)[i * n_actions + a])
                        : reinterpret_cast<const float*>(probs)[i * n_actions + a];
        total += p[a];
    }
    const float target = u * total;            // probs need not be normalised exactly (bf16 softmax)
    float cum = 0.f;
    int pick = n_actions - 1;
    bool found = false;
#pragma unroll
    for (int a = 0; a < 8; ++a) {              // smallest a with target < p[0] + ... + p[a]
        cum += p[a];
        if (!found && a < n_actions && target < cum) { pick = a; found = true; }
    }
    actions[i] = (uint8_t)pick;
}

// Egocentric proximity observations (wab_env.py:637-667, :951-958): for the five squares the ostrich can reach next
// (up, right, down, left, stay) the proximity max_distance - taxicab distance (clipped to [0, max_distance]) of the
// nearest wolf and of the nearest bush with food among EVERY cell seen this episode. One warp per env, on the state
// as stored after the last step: wolves go over the lanes; the cells of the taxicab-11 diamond around the ostrich go
// over the lanes too — inside the window the occupancy mask answers, outside it a cell counts iff some earlier
// position of this episode had it in view (position history, st.hist), its procedural draw makes it a bush and the
// depletion log has not emptied it. No wolf (no bush) at all: the reference substitutes distance 0 (:648, :664).
__global__ void __launch_bounds__(128) wab_ego_kernel(const __grid_constant__ Params P, const StatePtrs st, uint8_t* __restrict__ out10) {
    __shared__ uint32_t hs[4][1025];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t idx = (int64_t)blockIdx.x * 4 + warp, n = st.n;
    if (idx >= n) return;
    constexpr int MAXD = VIEW / 2 + VIEW / 2 + 1;
    const uint32_t pos = st.pos[idx], misc = st.misc[idx], nl = st.nlog[idx];
    const int32_t x = unpack_x(pos), y = unpack_y(pos);
    const uint32_t nw = ((misc >> 11) & 15u) | (((nl >> 9) & 7u) << 4), dep = (misc >> 15) & 1u, nlog = nl & 0xFFu;
    int32_t turn = (int32_t)(misc >> 16);
    if (turn > st.hist_len - 1) turn = st.hist_len - 1;
    const uint4 mb = st.bush[idx];
    const uint32_t m[4] = {mb.x, mb.y, mb.z, mb.w};
    const uint2 bk = st.bkey[idx];
    const uint32_t logsig = st.logsig[idx];
    for (int t = lane; t <= turn; t += 32) hs[warp][t] = t == 0 ? 0u : st.hist[(int64_t)t * n + idx];   // turn 0 is (0, 0)
    __syncwarp();
    const int32_t cx[5] = {x, x + 1, x, x - 1, x}, cy[5] = {y + 1, y, y - 1, y, y};       // generate_potential_actions :76-82
    int32_t dw[5], db[5];
#pragma unroll
    for (int a = 0; a < 5; ++a) { dw[a] = 1 << 20; db[a] = 1 << 20; }
    for (uint32_t k = (uint32_t)lane; k < nw; k += 32) {
        const uint32_t p = st.wolves[(int64_t)k * n + idx];
        const int32_t wx = unpack_x(p), wy = unpack_y(p);
#pragma unroll
        for (int a = 0; a < 5; ++a) dw[a] = min(dw[a], abs(cx[a] - wx) + abs(cy[a] - wy));
    }
    constexpr int SPAN = 2 * MAXD + 1;                       // 23 x 23 box around the ostrich, diamond inside
    for (int c = lane; c < SPAN * SPAN; c += 32) {
        const int32_t ddx = c / SPAN - MAXD, ddy = c % SPAN - MAXD;
        if (abs(ddx) + abs(ddy) > MAXD) continue;            // farther than 10 from all five squares: proximity 0 anyway
        const int32_t px = x + ddx, py = y + ddy;
        bool has;
        if (abs(ddx) <= HALF && abs(ddy) <= HALF) {
            const int bit = 11 * (HALF - ddx) + (HALF - ddy);     // [5 - (objx - x)][5 - (objy - y)]
            has = (m[bit >> 5] >> (bit & 31)) & 1u;
        } else {
            bool seen = false;
            for (int t = 0; t <= turn && !seen; ++t) {
                const uint32_t h = hs[warp][t];
                seen = abs(px - unpack_x(h)) <= HALF && abs(py - unpack_y(h)) <= HALF;
            }
            has = false;
            if (seen && P.n_bush_thr > 0) {
                const uint32_t word = bush_word_rare(pack_xy(px >> 1, py >> 1) ^ bk.x, bk.y, P.rk2[0], bush_lane(px, py));
                has = word >= P.thr_bush1;
                if (has && dep && (logsig & cell_sig(pack_xy(px, py)))) {
                    const uint32_t cell = pack_xy(px, py);
                    for (uint32_t l = 0; l < nlog; ++l)
                        if (st.logcell[(int64_t)l * n + idx] == cell) { has = alive_after(P, word, (uint32_t)st.logcnt[(int64_t)l * n + idx]); break; }
                }
            }
        }
        if (has) {
#pragma unroll
            for (int a = 0; a < 5; ++a) db[a] = min(db[a], abs(cx[a] - px) + abs(cy[a] - py));
        }
    }
    uint32_t res = 0;
#pragma unroll
    for (int a = 0; a < 5; ++a) {
        int32_t w = __reduce_min_sync(FULL, dw[a]), b = __reduce_min_sync(FULL, db[a]);
        if (w >= (1 << 20)) w = 0;                            // pd.Series([0] * 5), :648
        if (b >= (1 << 20)) b = 0;                            // :664
        const int32_t pw = max(0, min(MAXD, MAXD - w)), pb = max(0, min(MAXD, MAXD - b));
        if (lane == a) res = (uint32_t)pw;
        if (lane == 5 + a) res = (uint32_t)pb;
    }
    if (lane < 10) out10[idx * 10 + lane] = (uint8_t)res;
}

__global__ void wab_philox_kernel(const __grid_constant__ Params P, const uint32_t* __restrict__ ctr, int64_t n,
                                  uint32_t* __restrict__ outw) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t w[4];
    philox(P, ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], w);
    outw[4 * i] = w[0]; outw[4 * i + 1] = w[1]; outw[4 * i + 2] = w[2]; outw[4 * i + 3] = w[3];
}

}  // namespace

#include "wab_generic.cuh"

namespace {

// ---------------------------------------------------------------------------------------- host
thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
    return fail(WAB_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define WAB_CUDA(call)                                         \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);  \
    } while (0)

void fill_round_keys2(Params2& P, uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) { P.rk0[r] = k0; P.rk1[r] = k1; k0 += PHILOX_W0; k1 += PHILOX_W1; }
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

struct WabVec {
    WabConfig cfg;
    Params P;
    StatePtrs st;
    int device;
    int64_t n;
    void* slab;
    uint32_t* d_thr;
    // device staging for the host-buffer entry points
    uint8_t* stage;
    size_t stage_bytes;
    int64_t stat_rows; // rows of st.wstats
    uint32_t* d_hist; // position history of every env's current episode (egocentric observations), or null
    bool generic;     // viewport other than 11 x 11 or spawn margin other than 1: warp-per-env kernels of wab_generic.cuh
    GenGeo geo;
    int64_t obs_bytes; // 3 * width * height
    int lpe;          // lanes per env chosen at create (see pick_lpe)
    int mb;           // CTAs per SM the thread-per-env kernel is built for (see pick_mb)
    int n_sm;         // multiprocessors of the device
    uint8_t* d_features;   // bound feature output, or null
    // host-buffer step as one CUDA graph (H2D actions -> step kernel -> D2H block), rebuilt when the pointers change
    cudaStream_t host_stream;
    cudaGraphExec_t host_graph;
    const void* g_actions; void* g_block; const void* g_features;
    bool graph_unsupported;
    int host_mapped;   // -1 unknown, 0 staged copies, 1 kernel writes the pinned host block directly
    bool started;      // reset or loaded once: the replica layout is fixed from then on
    const void* m_actions; const void* m_block;        // host buffer pair whose device aliases are cached below
    const uint8_t* m_dactions; uint8_t* m_dblock;
    uint64_t fp_config;    // fingerprint of config, bush thresholds, seed and kernel kind (wab_state.cuh; ego folded in on query)
    uint8_t* d_zero_mask;  // u8[N] zeros: a reset that resets nothing re-emits every env's observation (after a state load)
};

namespace {

template <int LPE> size_t smem_bytes_for(const Params& P) {
    return sizeof(uint32_t) * ((size_t)P.wolf_cap * Geo<LPE>::EPB + (size_t)Geo<LPE>::STREAM + 512);
}
template <bool F64, int LPE>
void launch_step_t(const WabVec* h, const uint8_t* a, int T, const OutPtrs& out, cudaStream_t s);
template <bool F64, int LPE>
void launch_reset_t(const WabVec* h, const uint8_t* mask, const OutPtrs& out, cudaStream_t s);
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int check_ptr_align(const void* p, const char* name) {
    if (((uintptr_t)p & 15u) != 0) return fail(WAB_E_CONFIG, std::string(name) + " must be 16-byte aligned");
    return WAB_OK;
}

// Kernel launch with the programmatic-stream-serialization attribute: back-to-back launches on a stream (or the kernel
// nodes of a captured graph) overlap the next launch's scheduling and prologue with the tail of the previous one; the
// kernels order themselves with griddepcontrol.wait. WAB_PDL=0 switches the attribute off (A/B runs).
bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("WAB_PDL"); return !(e && atoi(e) == 0); }();
    return on;
}
template <typename... KArgs, typename... Args>
void launch_pdl(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// // WAB_PIPE: 0 = never, 1 (default) = where it pays (see launch_step_t), 2 = always (tests, A/B runs).
int pipe_mode() { const char* e = getenv("WAB_PIPE"); return e ? atoi(e) : 1; }
bool use_pipeline(const WabVec* h, int lpe, int T) {
    if (h->generic || lpe <= 1 || T < 4 || pipe_mode() == 0) return false;
    const int64_t epw = 32 / lpe, rule_warps = (h->n + epw - 1) / epw;
    return pipe_mode() == 2 || rule_warps <= 8 * (int64_t)h->n_sm;
}
template <bool F64, int LPE>
void launch_step_t(const WabVec* h, const uint8_t* a, int T, const OutPtrs& out, cudaStream_t s) {
    const unsigned grid = (unsigned)((h->n + Geo<LPE>::EPB - 1) / Geo<LPE>::EPB);
    if constexpr (LPE > 1) {
        // two-warp pipeline (rules in one warp, publication in the other) while the batch leaves issue slots free: up to
        // 8 rule warps per SM. Same-box A/B (profiles/r2j_pipe_ab.txt): 4,096 envs at LPE 8 (6.9 rule warps per SM)
        // 1.76e9 -> 1.97e9 env-steps/s, 2,048 at LPE 16 1.05e9 -> 1.21e9; 8,192 at LPE 8 (13.8 per SM) 2.74e9 -> 2.06e9.
        if (use_pipeline(h, LPE, T)) {
            const size_t smem = sizeof(uint32_t) * (size_t)PipeGeo<LPE>::PAIRS * (size_t)PipeGeo<LPE>::pair_words(h->P.wolf_cap);
            const int64_t groups = (h->n + PipeGeo<LPE>::EPW - 1) / PipeGeo<LPE>::EPW;
            const unsigned pgrid = (unsigned)((groups + PipeGeo<LPE>::PAIRS - 1) / PipeGeo<LPE>::PAIRS);
            launch_pdl(wab_step_pipe_kernel<F64, LPE>, pgrid, PipeGeo<LPE>::THREADS, smem, s, h->P, h->st, a, T, out);
            return;
        }
    }
    if (LPE == 1 && h->mb == 7)
        launch_pdl(wab_step_kernel<F64, LPE, LPE == 1 ? 7 * kMbScale : Geo<LPE>::MIN_BLOCKS>, grid, Geo<LPE>::THREADS, smem_bytes_for<LPE>(h->P), s, h->P, h->st, a, T, out);
    else if (LPE == 1 && h->mb == 8)
        launch_pdl(wab_step_kernel<F64, LPE, LPE == 1 ? 8 * kMbScale : Geo<LPE>::MIN_BLOCKS>, grid, Geo<LPE>::THREADS, smem_bytes_for<LPE>(h->P), s, h->P, h->st, a, T, out);
    else
        launch_pdl(wab_step_kernel<F64, LPE>, grid, Geo<LPE>::THREADS, smem_bytes_for<LPE>(h->P), s, h->P, h->st, a, T, out);
}
template <bool F64, int LPE>
void launch_reset_t(const WabVec* h, const uint8_t* mask, const OutPtrs& out, cudaStream_t s) {
    const unsigned grid = (unsigned)((h->n + Geo<LPE>::EPB - 1) / Geo<LPE>::EPB);
    launch_pdl(wab_reset_kernel<F64, LPE>, grid, Geo<LPE>::THREADS, smem_bytes_for<LPE>(h->P), s, h->P, h->st, mask, out);
}
// Lanes per env: the largest LPE whose whole grid is co-resident (one wave) on this device, so that a
// small batch spreads over all SMs and shortens its per-step critical path; large batches use the
// thread-per-env kernel, which wastes no issue slots. WAB_LPE overrides (tests, tuning).
template <int LPE>
bool fits_one_wave(const WabVec* h, int n_sm) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wab_step_kernel<false, LPE>, Geo<LPE>::THREADS,
                                                      smem_bytes_for<LPE>(h->P)) != cudaSuccess)
        return false;
    const int64_t grid = (h->n + Geo<LPE>::EPB - 1) / Geo<LPE>::EPB;
    return grid <= (int64_t)per_sm * n_sm;
}
int pick_lpe(const WabVec* h) {
    if (const char* e = getenv("WAB_LPE")) {
        const int v = atoi(e);
        if (v == 1 || v == 4 || v == 8 || v == 16 || v == 32) return v;
    }
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, h->device);
    // measured on B200 (profiles/r1_tune_lpe.jsonl): the best variant keeps 32k-64k threads in flight, and more than
    // 8 lanes per env only pays for very small batches (a step has 6 independent Philox calls to share out)
    const int64_t n = h->n;
    if (n * 32 <= 32768 && fits_one_wave<32>(h, n_sm)) return 32;
    if (n * 16 <= 32768 && fits_one_wave<16>(h, n_sm)) return 16;
    if (n * 8 <= 65536 && fits_one_wave<8>(h, n_sm)) return 8;
    if (n * 4 <= 65536 && fits_one_wave<4>(h, n_sm)) return 4;
    return 1;
}

// Thread-per-env batches of a little more than one wave of 6 CTAs per SM (113,664 envs on 148 SMs) run as ONE wave
// of 7 or 8 CTAs per SM with a tighter register cap: measured at 131,072 envs 1.05e10 (7) / 1.03e10 (8) against
// 0.94e10 env-steps/s (6); with two or more waves the cap only costs (profiles/r1f_wave_quantization.txt).
int pick_mb(const WabVec* h) {
    if (const char* e = getenv("WAB_MB")) {
        const int v = atoi(e);
        if (v >= 6 && v <= 8) return v;
    }
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, h->device);
    const int64_t grid = (h->n + Geo<1>::EPB - 1) / Geo<1>::EPB;
    for (int mb = 6; mb <= 8; ++mb)
        if (grid <= (int64_t)mb * kMbScale * n_sm) return mb;
    return 6;
}

#define WAB_DISPATCH(FN, ...) WAB_DISPATCH_LPE(h->lpe, FN, __VA_ARGS__)
#define WAB_DISPATCH_LPE(LPE_, FN, ...)                                                        \
    do {                                                                                       \
        const bool f64__ = h->cfg.food_mode == WAB_FOOD_F64;                                   \
        switch (LPE_) {                                                                        \
            case 32: f64__ ? FN<true, 32>(__VA_ARGS__) : FN<false, 32>(__VA_ARGS__); break;    \
            case 16: f64__ ? FN<true, 16>(__VA_ARGS__) : FN<false, 16>(__VA_ARGS__); break;    \
            case 8: f64__ ? FN<true, 8>(__VA_ARGS__) : FN<false, 8>(__VA_ARGS__); break;       \
            case 4: f64__ ? FN<true, 4>(__VA_ARGS__) : FN<false, 4>(__VA_ARGS__); break;       \
            default: f64__ ? FN<true, 1>(__VA_ARGS__) : FN<false, 1>(__VA_ARGS__); break;      \
        }                                                                                      \
    } while (0)

// d_grids may be NULL for FEATURES-ONLY stepping: a PragmaticObsWrapper feature buffer is bound (wab_vec_bind_features) and
// the caller — the reference's actor-critic consumes nothing else (actor_critic.py:42, :188) — does not want the 363-byte
// one-hot grids materialised in HBM. Specialised 11 x 11 kernels only.
int check_grids(const WabVec* h, const uint8_t* d_grids) {
    if (!d_grids) {
        if (h->generic || !h->d_features) return fail(WAB_E_NULL, "d_grids may only be null with a bound feature buffer (wab_vec_bind_features)");
        return WAB_OK;
    }
    return check_ptr_align(d_grids, "d_grids");
}

int launch_step(WabVec* h, int n_steps, const uint8_t* d_actions, const WabObs& obs, float* d_reward,
                uint8_t* d_done, uint8_t* d_info, cudaStream_t s, int lpe = 0) {
    OutPtrs out{obs.d_grids, obs.d_food, obs.d_role, obs.d_status, d_reward, d_done, d_info, h->d_features};
    if (h->generic) {
        const unsigned grid = (unsigned)((h->n + GEN_WARPS - 1) / GEN_WARPS);
        const size_t smem = sizeof(uint32_t) * (size_t)GEN_WARPS * (size_t)h->geo.warp_words;
        if (h->cfg.food_mode == WAB_FOOD_F64)
            launch_pdl(wab_generic_step_kernel<true>, grid, GEN_WARPS * 32, smem, s, h->P, h->st, h->geo, d_actions, n_steps, out);
        else
            launch_pdl(wab_generic_step_kernel<false>, grid, GEN_WARPS * 32, smem, s, h->P, h->st, h->geo, d_actions, n_steps, out);
        WAB_CUDA(cudaGetLastError());
        return WAB_OK;
    }
    WAB_DISPATCH_LPE(lpe ? lpe : h->lpe, launch_step_t, h, d_actions, n_steps, out, s);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int ensure_stage(WabVec* h, size_t bytes) {
    if (h->stage_bytes >= bytes) return WAB_OK;
    if (h->stage) cudaFree(h->stage);
    if (h->host_graph) { cudaGraphExecDestroy(h->host_graph); h->host_graph = nullptr; }
    h->stage = nullptr; h->stage_bytes = 0;
    WAB_CUDA(cudaMalloc(&h->stage, bytes));
    h->stage_bytes = bytes;
    return WAB_OK;
}

struct StageLayout { size_t actions, grids, food, role, status, reward, done, info, total; };
StageLayout stage_layout(int64_t n, int64_t obs_bytes = OBS_BYTES) {
    StageLayout L;
    size_t o = 0;
    L.actions = o; o = align_up(o + (size_t)n, 256);
    L.grids = o; o = align_up(o + (size_t)n * (size_t)obs_bytes, 256);
    L.food = o; o = align_up(o + (size_t)n, 256);
    L.role = o; o = align_up(o + (size_t)n, 256);
    L.status = o; o = align_up(o + (size_t)n, 256);
    L.reward = o; o = align_up(o + (size_t)n * 4, 256);
    L.done = o; o = align_up(o + (size_t)n, 256);
    L.info = o; o = align_up(o + (size_t)n, 256);
    L.total = o;
    return L;
}

}  // namespace

extern "C" {

const char* wab_last_error(void) { return g_err.c_str(); }
int wab_abi_version(void) { return WAB_ABI_VERSION; }

#if defined(WAB_PIPE_CLOCKS)
// Probe build only (tools/pipe_clocks.py): copy the current device's PC_N + PP_N probe totals to `out`, then zero them
// if `clear`. Synchronises the device.
int wab_pipe_clocks_read(unsigned long long* out, int clear) {
    if (cudaDeviceSynchronize() != cudaSuccess ||
        cudaMemcpyFromSymbol(out, wab_pipe_clocks_buf, sizeof(wab_pipe_clocks_buf)) != cudaSuccess)
        return fail(WAB_E_CUDA, "wab_pipe_clocks_read failed");
    if (clear) {
        static const unsigned long long zero[PC_N + PP_N] = {};
        if (cudaMemcpyToSymbol(wab_pipe_clocks_buf, zero, sizeof(zero)) != cudaSuccess)
            return fail(WAB_E_CUDA, "wab_pipe_clocks_read failed");
    }
    return WAB_OK;
}
#endif

int wab_vec_create(const WabConfig* cfg, const uint32_t* bush_thr, int32_t n_bush_thr, int64_t n_envs,
                   uint64_t seed, uint64_t env_id_base, int32_t device, WabVec** out) {
    if (!cfg || !out || (n_bush_thr > 0 && !bush_thr)) return fail(WAB_E_NULL, "null argument");
    *out = nullptr;
    if (int rc = validate_config(cfg, n_bush_thr, n_envs, g_err)) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(WAB_E_NO_DEVICE, "no CUDA device: wab_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(WAB_E_CONFIG, "bad device ordinal");
    DeviceGuard guard(device);

    WabVec* h = new (std::nothrow) WabVec();
    if (!h) return fail(WAB_E_CUDA, "out of host memory");
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg; h->device = device; h->n = n_envs; h->host_mapped = -1;
    h->generic = cfg->width != VIEW || cfg->height != VIEW || cfg->wolf_spawn_margin != 1 || getenv("WAB_GENERIC") != nullptr;
    h->geo = make_gen_geo(cfg->width, cfg->height, cfg->wolf_spawn_margin, cfg->wolf_cap);
    h->obs_bytes = 3 * (int64_t)cfg->width * cfg->height;

    Params& P = h->P;
    params_from_config(*cfg, bush_thr, n_bush_thr, seed, env_id_base, P);

    // one slab, every array 256-byte aligned
    const size_t n = (size_t)n_envs;
    size_t o = 0;
    const size_t o_pos = o; o = align_up(o + 4 * n, 256);
    const size_t o_misc = o; o = align_up(o + 4 * n, 256);
    const size_t o_ep = o; o = align_up(o + 4 * n, 256);
    const size_t o_bush = o; o = align_up(o + 16 * n, 256);
    const size_t o_nlog = o; o = align_up(o + 2 * n, 256);
    const size_t o_lsig = o; o = align_up(o + 4 * n, 256);
    const size_t o_bkey = o; o = align_up(o + 8 * n, 256);
    const size_t o_food = o; o = align_up(o + 8 * n, 256);
    const size_t o_wolves = o; o = align_up(o + 4 * n * (size_t)cfg->wolf_cap, 256);
    const size_t o_lcell = o; o = align_up(o + 4 * n * (size_t)cfg->log_cap, 256);
    const size_t o_lcnt = o; o = align_up(o + n * (size_t)cfg->log_cap, 256);
    const size_t o_stats = o; o = align_up(o + 64, 256);
    // one statistics row per warp of the largest grid this handle launches: its lanes-per-env variant, or thread per
    // env (which the mapped host path uses whatever the handle's variant is)
    h->n_sm = 148;
    cudaDeviceGetAttribute(&h->n_sm, cudaDevAttrMultiProcessorCount, device);
    h->lpe = pick_lpe(h);
    h->mb = pick_mb(h);
    auto warps_of = [n](size_t lpe) {
        const size_t threads = lpe == 1 ? (size_t)WAB_THREADS_LPE1 : (size_t)WAB_THREADS_LPEN, epb = threads / lpe;
        return (n + epb - 1) / epb * (threads / 32);
    };
    const size_t stat_rows = h->generic ? (n + GEN_WARPS - 1) / GEN_WARPS * GEN_WARPS
                                        : (warps_of(1) > warps_of((size_t)h->lpe) ? warps_of(1) : warps_of((size_t)h->lpe));
    const size_t o_wstats = o; o = align_up(o + 64 * stat_rows, 256);
    cudaError_t e = cudaMalloc(&h->slab, o);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaMalloc(state)"); }
    uint8_t* base = (uint8_t*)h->slab;
    e = cudaMemset(base, 0, o);
    if (e == cudaSuccess) e = cudaMemset(base + o_ep, 0xFF, 4 * n);   // episode -1: first reset -> 0
    if (e == cudaSuccess && n_bush_thr > 0) {
        e = cudaMalloc(&h->d_thr, sizeof(uint32_t) * (size_t)n_bush_thr);
        if (e == cudaSuccess)
            e = cudaMemcpy(h->d_thr, bush_thr, sizeof(uint32_t) * (size_t)n_bush_thr, cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) { cudaFree(h->slab); if (h->d_thr) cudaFree(h->d_thr); delete h; return cuda_fail(e, "state init"); }
    P.bush_thr = h->d_thr;
    StatePtrs& st = h->st;
    st.pos = (uint32_t*)(base + o_pos); st.misc = (uint32_t*)(base + o_misc); st.episode = (uint32_t*)(base + o_ep);
    st.bush = (uint4*)(base + o_bush); st.nlog = (uint16_t*)(base + o_nlog); st.logsig = (uint32_t*)(base + o_lsig); st.bkey = (uint2*)(base + o_bkey); st.food = (double*)(base + o_food);
    st.wolves = (uint32_t*)(base + o_wolves); st.logcell = (uint32_t*)(base + o_lcell); st.logcnt = base + o_lcnt;
    st.stats = (unsigned long long*)(base + o_stats); st.n = n_envs;
    st.wstats = (unsigned long long*)(base + o_wstats); h->stat_rows = (int64_t)stat_rows;
    h->fp_config = config_fingerprint(*cfg, bush_thr, n_bush_thr, seed, h->generic);
    *out = h;
    return WAB_OK;
}

void wab_vec_destroy(WabVec* h) {
    if (!h) return;
    DeviceGuard guard(h->device);
    if (h->slab) cudaFree(h->slab);
    if (h->d_hist) cudaFree(h->d_hist);
    if (h->d_thr) cudaFree(h->d_thr);
    if (h->d_zero_mask) cudaFree(h->d_zero_mask);
    if (h->stage) cudaFree(h->stage);
    if (h->host_graph) cudaGraphExecDestroy(h->host_graph);
    if (h->host_stream) cudaStreamDestroy(h->host_stream);
    delete h;
}

int64_t wab_vec_num_envs(const WabVec* h) { return h ? h->n : 0; }
int wab_vec_kernel_kind(const WabVec* h) { return h && h->generic ? 1 : 0; }
int wab_vec_lanes_per_env(const WabVec* h) { return h ? (h->generic ? 32 : h->lpe) : 0; }
int wab_vec_step_many_pipelined(const WabVec* h, int32_t n_steps) { return h && use_pipeline(h, h->lpe, n_steps) ? 1 : 0; }

int wab_vec_reset(WabVec* h, const uint8_t* d_mask, WabObs obs, void* stream) {
    if (!h || !obs.d_food || !obs.d_role || !obs.d_status) return fail(WAB_E_NULL, "null argument");
    if (int rc = check_grids(h, obs.d_grids)) return rc;
    DeviceGuard guard(h->device);
    h->started = true;
    OutPtrs out{obs.d_grids, obs.d_food, obs.d_role, obs.d_status, nullptr, nullptr, nullptr, h->d_features};
    cudaStream_t s = (cudaStream_t)stream;
    if (h->generic) {
        const unsigned grid = (unsigned)((h->n + GEN_WARPS - 1) / GEN_WARPS);
        const size_t smem = sizeof(uint32_t) * (size_t)GEN_WARPS * (size_t)h->geo.warp_words;
        if (h->cfg.food_mode == WAB_FOOD_F64)
            launch_pdl(wab_generic_reset_kernel<true>, grid, GEN_WARPS * 32, smem, s, h->P, h->st, h->geo, d_mask, out);
        else
            launch_pdl(wab_generic_reset_kernel<false>, grid, GEN_WARPS * 32, smem, s, h->P, h->st, h->geo, d_mask, out);
        WAB_CUDA(cudaGetLastError());
        return WAB_OK;
    }
    WAB_DISPATCH(launch_reset_t, h, d_mask, out, s);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_vec_step(WabVec* h, const uint8_t* d_actions, WabObs obs, float* d_reward, uint8_t* d_done,
                 uint8_t* d_info, void* stream) {
    if (!h || !d_actions || !obs.d_food || !obs.d_role || !obs.d_status || !d_reward || !d_done)
        return fail(WAB_E_NULL, "null argument");
    if (int rc = check_grids(h, obs.d_grids)) return rc;
    DeviceGuard guard(h->device);
    return launch_step(h, 1, d_actions, obs, d_reward, d_done, d_info, (cudaStream_t)stream);
}

int wab_vec_step_many(WabVec* h, int32_t n_steps, const uint8_t* d_actions, WabObs obs, float* d_reward,
                      uint8_t* d_done, uint8_t* d_info, void* stream) {
    if (!h || !d_actions || !obs.d_food || !obs.d_role || !obs.d_status || !d_reward || !d_done)
        return fail(WAB_E_NULL, "null argument");
    if (n_steps < 1 || n_steps > 65535) return fail(WAB_E_CONFIG, "n_steps must be in [1, 65535]");
    if (int rc = check_grids(h, obs.d_grids)) return rc;
    DeviceGuard guard(h->device);
    return launch_step(h, n_steps, d_actions, obs, d_reward, d_done, d_info, (cudaStream_t)stream);
}

int wab_vec_step_host(WabVec* h, const uint8_t* h_actions, uint8_t* h_grids, uint8_t* h_food, uint8_t* h_role,
                      uint8_t* h_status, float* h_reward, uint8_t* h_done, uint8_t* h_info, void* stream) {
    if (!h || !h_actions || !h_grids || !h_food || !h_role || !h_status || !h_reward || !h_done)
        return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const StageLayout L = stage_layout(h->n, h->obs_bytes);
    if (int rc = ensure_stage(h, L.total)) return rc;
    uint8_t* b = h->stage;
    const size_t n = (size_t)h->n;
    WAB_CUDA(cudaMemcpyAsync(b + L.actions, h_actions, n, cudaMemcpyHostToDevice, s));
    WabObs obs{b + L.grids, b + L.food, b + L.role, b + L.status};
    if (int rc = launch_step(h, 1, b + L.actions, obs, (float*)(b + L.reward), b + L.done, b + L.info, s)) return rc;
    WAB_CUDA(cudaMemcpyAsync(h_grids, b + L.grids, n * (size_t)h->obs_bytes, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_food, b + L.food, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_role, b + L.role, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_status, b + L.status, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_reward, b + L.reward, n * 4, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_done, b + L.done, n, cudaMemcpyDeviceToHost, s));
    if (h_info) WAB_CUDA(cudaMemcpyAsync(h_info, b + L.info, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaStreamSynchronize(s));
    return WAB_OK;
}

int wab_vec_host_block_layout(const WabVec* h, int64_t* offsets7, int64_t* total_bytes) {
    if (!h || !offsets7 || !total_bytes) return fail(WAB_E_NULL, "null argument");
    const StageLayout L = stage_layout(h->n, h->obs_bytes);
    const size_t v[7] = {L.grids, L.food, L.role, L.status, L.reward, L.done, L.info};
    for (int k = 0; k < 7; ++k) offsets7[k] = (int64_t)(v[k] - L.grids);
    *total_bytes = (int64_t)(L.total - L.grids);
    return WAB_OK;
}

int wab_vec_step_host_packed(WabVec* h, const uint8_t* h_actions, uint8_t* h_block, void* stream) {
    if (!h || !h_actions || !h_block) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const StageLayout L = stage_layout(h->n, h->obs_bytes);
    if (int rc = ensure_stage(h, L.total)) return rc;
    uint8_t* b = h->stage;
    WabObs obs{b + L.grids, b + L.food, b + L.role, b + L.status};
    // Zero-copy path (batches up to 16k envs, where a step is latency- rather than PCIe-bandwidth-bound): the
    // thread-per-env kernel — whose warps own 16-byte-aligned slabs, so every store is a full 16-byte one — reads the
    // actions from, and streams its outputs into, the caller's pinned (hence device-mapped) host buffers; no staging
    // copy, and the transfer overlaps the step. Measured (profiles/r1_e2e_paths.txt): 52.7 vs 60.2 us per step at
    // 4,096 envs; the copy engine wins from 32k envs up. WAB_HOST_MAPPED=0 forces the staged path, any other value the
    // mapped one.
    if (h->host_mapped < 0) {
        const char* e = getenv("WAB_HOST_MAPPED");
        h->host_mapped = e ? atoi(e) != 0 : h->n <= 16384;
    }
    if (h->host_mapped) {
        if (h->m_actions != h_actions || h->m_block != h_block) {      // resolve the device aliases once per buffer pair
            cudaPointerAttributes pa, pb;
            h->m_actions = h_actions; h->m_block = h_block; h->m_dactions = nullptr; h->m_dblock = nullptr;
            // the kernel's 16-byte observation stores align themselves to any address, its f32 reward stores need the
            // block's 256-byte-aligned offsets to stay 4-byte aligned: a block that is not 16-byte aligned takes the staged path
            if (cudaPointerGetAttributes(&pa, h_actions) == cudaSuccess && cudaPointerGetAttributes(&pb, h_block) == cudaSuccess &&
                pa.type == cudaMemoryTypeHost && pb.type == cudaMemoryTypeHost && pa.devicePointer && pb.devicePointer &&
                ((uintptr_t)pb.devicePointer & 15u) == 0) {
                h->m_dactions = (const uint8_t*)pa.devicePointer; h->m_dblock = (uint8_t*)pb.devicePointer;
            } else {
                cudaGetLastError();                // pageable memory: staged copies below
            }
        }
        if (h->m_dblock) {
            uint8_t* m = h->m_dblock - L.grids;                        // block offsets are relative to L.grids
            WabObs mo{m + L.grids, m + L.food, m + L.role, m + L.status};
            if (int rc = launch_step(h, 1, h->m_dactions, mo, (float*)(m + L.reward), m + L.done, m + L.info, s, 1)) return rc;
            WAB_CUDA(cudaStreamSynchronize(s));
            return WAB_OK;
        }
    }
    // Fast path: the three operations replayed as one graph launch on a private stream (saves two API round trips
    // per step; needs pinned host buffers — anything else falls back to the plain sequence below).
    if (!h->graph_unsupported) {
        if (!h->host_stream && cudaStreamCreateWithFlags(&h->host_stream, cudaStreamNonBlocking) != cudaSuccess) {
            cudaGetLastError(); h->graph_unsupported = true;
        }
        if (!h->graph_unsupported && (!h->host_graph || h->g_actions != h_actions || h->g_block != h_block ||
                                      h->g_features != h->d_features)) {
            if (h->host_graph) { cudaGraphExecDestroy(h->host_graph); h->host_graph = nullptr; }
            cudaGraph_t graph = nullptr;
            bool ok = cudaStreamBeginCapture(h->host_stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            if (ok) {
                ok = cudaMemcpyAsync(b + L.actions, h_actions, (size_t)h->n, cudaMemcpyHostToDevice, h->host_stream) == cudaSuccess;
                ok = ok && launch_step(h, 1, b + L.actions, obs, (float*)(b + L.reward), b + L.done, b + L.info, h->host_stream) == WAB_OK;
                ok = ok && cudaMemcpyAsync(h_block, b + L.grids, L.total - L.grids, cudaMemcpyDeviceToHost, h->host_stream) == cudaSuccess;
                ok = (cudaStreamEndCapture(h->host_stream, &graph) == cudaSuccess) && ok && graph;
            }
            if (ok) ok = cudaGraphInstantiate(&h->host_graph, graph, 0) == cudaSuccess;
            if (graph) cudaGraphDestroy(graph);
            if (!ok) { cudaGetLastError(); h->host_graph = nullptr; h->graph_unsupported = true; }
            h->g_actions = h_actions; h->g_block = h_block; h->g_features = h->d_features;
        }
        if (h->host_graph) {
            WAB_CUDA(cudaStreamSynchronize(s));                 // order after the caller's earlier work
            WAB_CUDA(cudaGraphLaunch(h->host_graph, h->host_stream));
            WAB_CUDA(cudaStreamSynchronize(h->host_stream));
            return WAB_OK;
        }
    }
    WAB_CUDA(cudaMemcpyAsync(b + L.actions, h_actions, (size_t)h->n, cudaMemcpyHostToDevice, s));
    if (int rc = launch_step(h, 1, b + L.actions, obs, (float*)(b + L.reward), b + L.done, b + L.info, s)) return rc;
    WAB_CUDA(cudaMemcpyAsync(h_block, b + L.grids, L.total - L.grids, cudaMemcpyDeviceToHost, s));   // one transfer
    WAB_CUDA(cudaStreamSynchronize(s));
    return WAB_OK;
}

// The host-buffer entry points cache what they resolved for the caller's buffers (device aliases of pinned memory, the
// captured copy-step-copy graph) by host address. A buffer that is freed or unregistered must be forgotten first: another
// allocation at the same address would otherwise inherit a stale alias.
int wab_vec_forget_host_buffers(WabVec* h) {
    if (!h) return fail(WAB_E_NULL, "null handle");
    DeviceGuard guard(h->device);
    h->m_actions = nullptr; h->m_block = nullptr; h->m_dactions = nullptr; h->m_dblock = nullptr;
    h->g_actions = nullptr; h->g_block = nullptr; h->g_features = nullptr;
    if (h->host_graph) { cudaGraphExecDestroy(h->host_graph); h->host_graph = nullptr; }
    return WAB_OK;
}

int wab_vec_reset_host(WabVec* h, uint8_t* h_grids, uint8_t* h_food, uint8_t* h_role, uint8_t* h_status,
                       void* stream) {
    if (!h || !h_grids || !h_food || !h_role || !h_status) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    const StageLayout L = stage_layout(h->n, h->obs_bytes);
    if (int rc = ensure_stage(h, L.total)) return rc;
    uint8_t* b = h->stage;
    const size_t n = (size_t)h->n;
    WabObs obs{b + L.grids, b + L.food, b + L.role, b + L.status};
    if (int rc = wab_vec_reset(h, nullptr, obs, stream)) return rc;
    WAB_CUDA(cudaMemcpyAsync(h_grids, b + L.grids, n * (size_t)h->obs_bytes, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_food, b + L.food, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_role, b + L.role, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaMemcpyAsync(h_status, b + L.status, n, cudaMemcpyDeviceToHost, s));
    WAB_CUDA(cudaStreamSynchronize(s));
    return WAB_OK;
}

int wab_vec_stats(WabVec* h, int64_t* h_out8, int32_t clear, void* stream) {
    if (!h || !h_out8) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    wab_stats_reduce_kernel<<<8, 256, 0, s>>>(h->st.wstats, h->stat_rows, h->st.stats);
    WAB_CUDA(cudaGetLastError());
    WAB_CUDA(cudaMemcpyAsync(h_out8, h->st.stats, 64, cudaMemcpyDeviceToHost, s));
    if (clear) WAB_CUDA(cudaMemsetAsync(h->st.wstats, 0, 64 * (size_t)h->stat_rows, s));
    WAB_CUDA(cudaStreamSynchronize(s));
    return WAB_OK;
}

int wab_vec_stats_device(WabVec* h, int64_t* d_out8, void* stream) {
    if (!h || !d_out8) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    // totals straight into the caller's buffer (the handle's own totals are left alone: this call may run on a side
    // stream concurrently with wab_vec_stats)
    wab_stats_reduce_kernel<<<8, 256, 0, (cudaStream_t)stream>>>(h->st.wstats, h->stat_rows, (unsigned long long*)d_out8);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_vec_export_state(WabVec* h, int32_t* x, int32_t* y, double* food, int32_t* role, int32_t* status,
                         int32_t* turn, int64_t* episode, int32_t* n_wolves, int32_t* wolves_xy,
                         uint32_t* bush_mask, int32_t* n_log, int32_t* log_xyc, void* stream) {
    if (!h) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    WAB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    const size_t n = (size_t)h->n;
    const int wc = h->cfg.wolf_cap, lc = h->cfg.log_cap;
    uint32_t* pos = new uint32_t[n]; uint32_t* misc = new uint32_t[n]; uint32_t* ep = new uint32_t[n];
    uint32_t* bush = new uint32_t[4 * n]; uint16_t* nl = new uint16_t[n]; double* fd = new double[n];
    uint32_t* wv = new uint32_t[n * wc]; uint32_t* lcell = new uint32_t[n * lc]; uint8_t* lcnt = new uint8_t[n * lc];
    cudaError_t e = cudaMemcpy(pos, h->st.pos, 4 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(misc, h->st.misc, 4 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(ep, h->st.episode, 4 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(bush, h->st.bush, 16 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(nl, h->st.nlog, 2 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(fd, h->st.food, 8 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(wv, h->st.wolves, 4 * n * wc, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(lcell, h->st.logcell, 4 * n * lc, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(lcnt, h->st.logcnt, n * lc, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) {
        for (size_t i = 0; i < n; ++i) {
            const uint32_t m = misc[i];
            const int nw = (int)(((m >> 11) & 15u) | (((nl[i] >> 9) & 7u) << 4));
            if (x) x[i] = unpack_x(pos[i]);
            if (y) y[i] = unpack_y(pos[i]);
            if (food) food[i] = h->cfg.food_mode == WAB_FOOD_F64 ? fd[i] : (double)(m & 0xFFu) / h->cfg.food_obs_scale;
            if (role) role[i] = (int32_t)((m >> 8) & 1u);
            if (status) status[i] = (int32_t)((m >> 9) & 3u);
            if (turn) turn[i] = (int32_t)(m >> 16);
            if (episode) episode[i] = (int64_t)(int32_t)ep[i];
            if (n_wolves) n_wolves[i] = nw;
            if (wolves_xy)
                for (int k = 0; k < wc; ++k) {
                    const uint32_t p = wv[(size_t)k * n + i];
                    wolves_xy[(i * wc + k) * 2] = k < nw ? unpack_x(p) : 0;
                    wolves_xy[(i * wc + k) * 2 + 1] = k < nw ? unpack_y(p) : 0;
                }
            if (bush_mask) for (int w = 0; w < 4; ++w) bush_mask[4 * i + w] = bush[4 * i + w];
            if (n_log) n_log[i] = nl[i] & 0xFF;
            if (log_xyc)
                for (int k = 0; k < lc; ++k) {
                    const uint32_t c = lcell[(size_t)k * n + i];
                    const bool live = k < (int)(nl[i] & 0xFF);
                    log_xyc[(i * lc + k) * 3] = live ? unpack_x(c) : 0;
                    log_xyc[(i * lc + k) * 3 + 1] = live ? unpack_y(c) : 0;
                    log_xyc[(i * lc + k) * 3 + 2] = live ? (int32_t)lcnt[(size_t)k * n + i] : 0;
                }
        }
    }
    delete[] pos; delete[] misc; delete[] ep; delete[] bush; delete[] nl; delete[] fd;
    delete[] wv; delete[] lcell; delete[] lcnt;
    if (e != cudaSuccess) return cuda_fail(e, "export_state");
    return WAB_OK;
}

int wab_vec_enable_ego(WabVec* h) {
    if (!h) return fail(WAB_E_NULL, "null argument");
    if (h->d_hist) return WAB_OK;
    if (h->cfg.max_turns > 1023) return fail(WAB_E_UNSUPPORTED, "egocentric observations keep a position history of at most 1,023 turns");
    if (h->generic) return fail(WAB_E_UNSUPPORTED, "egocentric observations are implemented for the 11 x 11 viewport with spawn margin 1");
    DeviceGuard guard(h->device);
    const size_t len = (size_t)h->cfg.max_turns + 1;
    WAB_CUDA(cudaMalloc(&h->d_hist, 4 * len * (size_t)h->n));
    WAB_CUDA(cudaMemset(h->d_hist, 0, 4 * len * (size_t)h->n));
    h->st.hist = h->d_hist; h->st.hist_len = (int32_t)len;
    if (h->host_graph) { cudaGraphExecDestroy(h->host_graph); h->host_graph = nullptr; }   // captured with the old StatePtrs
    return WAB_OK;
}

int wab_vec_set_replicas(WabVec* h, int64_t n_replicas) {
    if (!h) return fail(WAB_E_NULL, "null argument");
    if (h->started) return fail(WAB_E_CONFIG, "call wab_vec_set_replicas before the first reset");
    if (n_replicas < 1 || h->n % n_replicas != 0) return fail(WAB_E_CONFIG, "n_replicas must divide n_envs");
    if (h->n > (int64_t)UINT32_MAX) return fail(WAB_E_CONFIG, "replicated handles hold fewer than 2^32 envs");
    h->P.replica_envs = n_replicas == 1 ? 0u : (uint32_t)(h->n / n_replicas);
    h->P.block_delta = 0u - h->P.replica_envs;                                            // block_stride 0
    if (h->host_graph) { cudaGraphExecDestroy(h->host_graph); h->host_graph = nullptr; }   // captured with the old Params
    return WAB_OK;
}

int wab_vec_set_blocks(WabVec* h, int64_t n_blocks, int64_t block_stride) {
    if (!h) return fail(WAB_E_NULL, "null argument");
    if (h->started) return fail(WAB_E_CONFIG, "call wab_vec_set_blocks before the first reset");
    if (n_blocks < 1 || h->n % n_blocks != 0) return fail(WAB_E_CONFIG, "n_blocks must divide n_envs");
    if (block_stride < 0 || (block_stride > 0 && block_stride < h->n / n_blocks))
        return fail(WAB_E_CONFIG, "block_stride must be 0 (replicas) or at least n_envs / n_blocks: the blocks' ids would overlap");
    if (h->n > (int64_t)UINT32_MAX) return fail(WAB_E_CONFIG, "blocked handles hold fewer than 2^32 envs");
    const int64_t c = h->n / n_blocks;
    if (block_stride > (int64_t)UINT32_MAX || (n_blocks - 1) * block_stride + c > ((int64_t)1 << 32))
        return fail(WAB_E_CONFIG, "a blocked handle's ids lie within 2^32 of env_id_base: (n_blocks - 1) block_stride + n_envs / n_blocks <= 2^32");
    h->P.replica_envs = n_blocks == 1 ? 0u : (uint32_t)c;
    h->P.block_delta = n_blocks == 1 ? 0u : (uint32_t)block_stride - (uint32_t)c;
    if (h->host_graph) { cudaGraphExecDestroy(h->host_graph); h->host_graph = nullptr; }   // captured with the old Params
    return WAB_OK;
}

int wab_vec_ego_proximities(WabVec* h, uint8_t* d_out10, void* stream) {
    if (!h || !d_out10) return fail(WAB_E_NULL, "null argument");
    if (!h->d_hist) return fail(WAB_E_CONFIG, "call wab_vec_enable_ego before the first reset");
    DeviceGuard guard(h->device);
    wab_ego_kernel<<<(unsigned)((h->n + 3) / 4), 128, 0, (cudaStream_t)stream>>>(h->P, h->st, d_out10);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_vec_bind_features(WabVec* h, uint8_t* d_features) {
    if (!h) return fail(WAB_E_NULL, "null argument");
    if (d_features && (h->cfg.width != VIEW || h->cfg.height != VIEW))
        return fail(WAB_E_UNSUPPORTED, "PragmaticObsWrapper features are implemented for the 11 x 11 viewport");
    if (((uintptr_t)d_features & 3u) != 0) return fail(WAB_E_CONFIG, "d_features must be 4-byte aligned");
    h->d_features = d_features;
    return WAB_OK;
}

int wab_vec_flat_dim(const WabVec* h) {
    return h ? 2 * (2 * 4 * (MAX_DISTANCE + 1) + 4 * 11) + 2 + ((int)h->cfg.food_obs_scale + 1) + 2 + 3 + CELLS : 0;
}

int wab_pragmatic_features(const uint8_t* d_grids, const uint8_t* d_food, const uint8_t* d_role, const uint8_t* d_status,
                           int64_t n, uint8_t* d_features, void* stream) {
    if (!d_grids || !d_food || !d_role || !d_status || !d_features) return fail(WAB_E_NULL, "null argument");
    if (((uintptr_t)d_features & 3u) != 0) return fail(WAB_E_CONFIG, "d_features must be 4-byte aligned");
    if (n <= 0) return WAB_OK;
    wab_features_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(d_grids, d_food, d_role, d_status, n, d_features);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_vec_flatten_features(WabVec* h, const uint8_t* d_features, int64_t n_rows, float* d_out, void* stream) {
    if (!h || !d_features || !d_out) return fail(WAB_E_NULL, "null argument");
    if (n_rows <= 0) return WAB_OK;
    DeviceGuard guard(h->device);
    const int64_t total = n_rows * wab_vec_flat_dim(h);
    wab_flatten_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, d_out);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_vec_flatten_features_noisy(WabVec* h, const uint8_t* d_features, int64_t n_rows, void* d_out, int32_t out_bf16,
                                   float noise_scale, const uint64_t* d_counter, void* stream) {
    if (!h || !d_features || !d_out) return fail(WAB_E_NULL, "null argument");
    if (n_rows <= 0) return WAB_OK;
    if (((uintptr_t)d_out & 15u) != 0) return fail(WAB_E_CONFIG, "d_out must be 16-byte aligned");
    DeviceGuard guard(h->device);
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, h->device);
    const int64_t want = (n_rows + 7) / 8;
    const unsigned grid = (unsigned)(want < (int64_t)n_sm * 8 ? want : (int64_t)n_sm * 8);
    const int food_dim = (int)h->cfg.food_obs_scale + 1;
    const unsigned long long* ctr = reinterpret_cast<const unsigned long long*>(d_counter);
    if (out_bf16)
        wab_flatten_noisy_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(h->P, d_features, n_rows, food_dim, d_out, noise_scale, ctr);
    else
        wab_flatten_noisy_kernel<0><<<grid, 256, 0, (cudaStream_t)stream>>>(h->P, d_features, n_rows, food_dim, d_out, noise_scale, ctr);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int64_t wab_policy_affine1_packed_bytes(void) { return (int64_t)TC_CHUNKS * 3 * TC_PART_BYTES; }

int wab_policy_affine1_prepare(const float* d_weight, int32_t in_dim, void* d_packed, void* stream) {
    if (!d_weight || !d_packed) return fail(WAB_E_NULL, "null argument");
    if (in_dim < 1 || in_dim > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, "wab_policy_affine1: the input is at most 512 columns wide");
    if (((uintptr_t)d_packed & 15u) != 0) return fail(WAB_E_CONFIG, "d_packed must be 16-byte aligned");
    const int total = TC_CHUNKS * TC_N * TC_KC;
    wab_affine1_prepare_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_weight, in_dim, reinterpret_cast<uint16_t*>(d_packed));
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_policy_affine1(WabVec* h, const uint8_t* d_features, int64_t n_rows, const void* d_packed, const float* d_bias,
                       float noise_scale, float leaky_slope, const uint64_t* d_counter, float* d_out, void* stream) {
    if (!h || !d_features || !d_packed || !d_bias || !d_out) return fail(WAB_E_NULL, "null argument");
    if (n_rows <= 0) return WAB_OK;
    if (((uintptr_t)d_out & 15u) != 0 || ((uintptr_t)d_packed & 15u) != 0 || ((uintptr_t)d_features & 3u) != 0)
        return fail(WAB_E_CONFIG, "d_out and d_packed must be 16-byte aligned, d_features 4-byte aligned");
    if (wab_vec_flat_dim(h) > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, "wab_policy_affine1: the input is at most 512 columns wide");
    DeviceGuard guard(h->device);
    static bool attr_set[64] = {false};
    if (h->device < 64 && !attr_set[h->device]) {
        WAB_CUDA(cudaFuncSetAttribute(wab_affine1_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_TOTAL));
        attr_set[h->device] = true;
    }
    const unsigned grid = (unsigned)((n_rows + TC_TILE_M - 1) / TC_TILE_M);
    wab_affine1_tc_kernel<0><<<grid, 256, TC_SMEM_TOTAL, (cudaStream_t)stream>>>(
        h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, reinterpret_cast<const uint4*>(d_packed), d_bias, noise_scale,
        leaky_slope, reinterpret_cast<const unsigned long long*>(d_counter), d_out, TrunkWeights());
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int64_t wab_policy_linear_packed_bytes(int32_t n_out, int32_t n_in) {
    const int64_t n_pad = (n_out + 15) / 16 * 16, k_pad = (n_in + T2_KC - 1) / T2_KC * T2_KC;
    return 3 * n_pad * k_pad * 2;
}

int wab_policy_linear_prepare(const float* d_weight, int32_t n_out, int32_t n_in, void* d_packed, void* stream) {
    if (!d_weight || !d_packed) return fail(WAB_E_NULL, "null argument");
    if (n_out < 1 || n_out > 256 || n_in < 1 || n_in > 512) return fail(WAB_E_UNSUPPORTED, "wab_policy_linear_prepare: at most 256 outputs and 512 inputs");
    if (((uintptr_t)d_packed & 15u) != 0) return fail(WAB_E_CONFIG, "d_packed must be 16-byte aligned");
    const int n_pad = (n_out + 15) / 16 * 16, k_pad = (n_in + T2_KC - 1) / T2_KC * T2_KC, total = n_pad * k_pad;
    wab_linear_prepare_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_weight, n_out, n_in, n_pad, k_pad, reinterpret_cast<uint16_t*>(d_packed));
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

static int policy_trunk_launch(WabVec* h, const uint8_t* d_features, int64_t n_rows, const void* d_packed1, const float* d_bias1,
                               const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                               float noise_scale, float leaky_slope, const uint64_t* d_counter, float* d_z3, void* stream,
                               const TrunkWeights* tail, bool greedy = false) {
    if (!h || !d_features || !d_packed1 || !d_bias1 || !d_packed2 || !d_bias2 || !d_packed3 || !d_bias3 || (!d_z3 && !tail)) return fail(WAB_E_NULL, "null argument");
    if (hidden2 != 150) return fail(WAB_E_UNSUPPORTED, "wab_policy_trunk is built for the reference's trunk 128 -> 150 -> 128 (actor_critic.py:59-61)");
    if (n_rows <= 0) return WAB_OK;
    if (((uintptr_t)d_z3 & 15u) != 0 || ((uintptr_t)d_packed1 & 15u) != 0 || ((uintptr_t)d_packed2 & 15u) != 0 || ((uintptr_t)d_packed3 & 15u) != 0 ||
        ((uintptr_t)d_features & 3u) != 0)
        return fail(WAB_E_CONFIG, "d_z3 and the packed weights must be 16-byte aligned, d_features 4-byte aligned");
    if (wab_vec_flat_dim(h) > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, "wab_policy_trunk: the input is at most 512 columns wide");
    DeviceGuard guard(h->device);
    static bool attr_set[64] = {false};
    if (h->device < 64 && !attr_set[h->device]) {
        WAB_CUDA(cudaFuncSetAttribute(wab_affine1_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_TOTAL));
        WAB_CUDA(cudaFuncSetAttribute(wab_affine1_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_TOTAL));
        WAB_CUDA(cudaFuncSetAttribute(wab_affine1_tc_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_TOTAL));
        WAB_CUDA(cudaFuncSetAttribute(wab_affine1_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_TOTAL));
        WAB_CUDA(cudaFuncSetAttribute(wab_affine1_tc_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_TOTAL));
        attr_set[h->device] = true;
    }
    TrunkWeights tw;
    if (tail) tw = *tail; else memset(&tw, 0, sizeof(tw));
    tw.w2 = reinterpret_cast<const uint4*>(d_packed2); tw.b2 = d_bias2; tw.w3 = reinterpret_cast<const uint4*>(d_packed3); tw.b3 = d_bias3; tw.n2 = hidden2;
    const unsigned grid = (unsigned)((n_rows + TC_TILE_M - 1) / TC_TILE_M);
    if (tail && tail->member_rows > 0 && greedy)
        wab_affine1_tc_kernel<5><<<grid, 256, TC_SMEM_TOTAL, (cudaStream_t)stream>>>(
            h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, reinterpret_cast<const uint4*>(d_packed1), d_bias1, noise_scale,
            leaky_slope, reinterpret_cast<const unsigned long long*>(d_counter), d_z3, tw);
    else if (tail && tail->member_rows > 0)
        wab_affine1_tc_kernel<4><<<grid, 256, TC_SMEM_TOTAL, (cudaStream_t)stream>>>(
            h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, reinterpret_cast<const uint4*>(d_packed1), d_bias1, noise_scale,
            leaky_slope, reinterpret_cast<const unsigned long long*>(d_counter), d_z3, tw);
    else if (tail && greedy)
        wab_affine1_tc_kernel<3><<<grid, 256, TC_SMEM_TOTAL, (cudaStream_t)stream>>>(
            h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, reinterpret_cast<const uint4*>(d_packed1), d_bias1, noise_scale,
            leaky_slope, reinterpret_cast<const unsigned long long*>(d_counter), d_z3, tw);
    else if (tail)
        wab_affine1_tc_kernel<2><<<grid, 256, TC_SMEM_TOTAL, (cudaStream_t)stream>>>(
            h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, reinterpret_cast<const uint4*>(d_packed1), d_bias1, noise_scale,
            leaky_slope, reinterpret_cast<const unsigned long long*>(d_counter), d_z3, tw);
    else
        wab_affine1_tc_kernel<1><<<grid, 256, TC_SMEM_TOTAL, (cudaStream_t)stream>>>(
            h->P, d_features, n_rows, (int)h->cfg.food_obs_scale + 1, reinterpret_cast<const uint4*>(d_packed1), d_bias1, noise_scale,
            leaky_slope, reinterpret_cast<const unsigned long long*>(d_counter), d_z3, tw);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_policy_trunk(WabVec* h, const uint8_t* d_features, int64_t n_rows, const void* d_packed1, const float* d_bias1,
                     const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                     float noise_scale, float leaky_slope, const uint64_t* d_counter, float* d_z3, void* stream) {
    if (!d_z3) return fail(WAB_E_NULL, "null argument");
    return policy_trunk_launch(h, d_features, n_rows, d_packed1, d_bias1, d_packed2, d_bias2, hidden2, d_packed3, d_bias3, noise_scale,
                               leaky_slope, d_counter, d_z3, stream, nullptr);
}

int wab_policy_forward(WabVec* h, const uint8_t* d_features, int64_t n_rows, const void* d_packed1, const float* d_bias1,
                       const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                       const float* d_w_heads, const float* d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                       float clamp_lo, float clamp_hi, uint64_t sample_seed, const uint64_t* d_counter, uint8_t* d_actions,
                       float* d_value, float* d_probs, float* d_logp, float* d_z3, void* stream) {
    if (!d_w_heads || !d_b_heads || !d_actions) return fail(WAB_E_NULL, "null argument");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_CONFIG, "n_actions must be in [1, 8]");
    TrunkWeights tw;
    memset(&tw, 0, sizeof(tw));
    uint32_t k0 = (uint32_t)sample_seed, k1 = (uint32_t)(sample_seed >> 32);
    for (int r = 0; r < 10; ++r) { tw.rk0[r] = k0; tw.rk1[r] = k1; k0 += PHILOX_W0; k1 += PHILOX_W1; }
    tw.w_heads = d_w_heads; tw.b_heads = d_b_heads; tw.n_actions = n_actions; tw.clamp_lo = clamp_lo; tw.clamp_hi = clamp_hi;
    tw.actions = d_actions; tw.value = d_value; tw.probs = d_probs; tw.logp = d_logp;
    return policy_trunk_launch(h, d_features, n_rows, d_packed1, d_bias1, d_packed2, d_bias2, hidden2, d_packed3, d_bias3, noise_scale,
                               leaky_slope, d_counter, d_z3, stream, &tw);
}

// wab_policy_forward_population (sample_seed given) and wab_policy_act_population (greedy, no seed): the checks they share,
// then MODE 4 or MODE 5 through policy_trunk_launch
static int policy_population_launch(const char* who, WabVec* h, const uint8_t* d_features, int32_t n_members,
                                    int64_t member_rows, const void* d_packed1, const float* d_bias1, const void* d_packed2,
                                    const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                                    const float* d_w_heads, const float* d_b_heads, int32_t n_actions, float noise_scale,
                                    float leaky_slope, float clamp_lo, float clamp_hi, const uint64_t* sample_seed,
                                    const uint64_t* d_counter, uint8_t* d_actions, float* d_value, float* d_probs, float* d_logp,
                                    float* d_z3, void* stream) {
    if (!d_w_heads || !d_b_heads || !d_actions) return fail(WAB_E_NULL, "null argument");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_CONFIG, "n_actions must be in [1, 8]");
    if (n_members < 1 || n_members > 64) return fail(WAB_E_CONFIG, std::string(who) + ": 1 <= n_members <= 64");
    if (member_rows < TC_TILE_M || member_rows % TC_TILE_M != 0)
        return fail(WAB_E_CONFIG, std::string(who) + ": member_rows must be a positive multiple of 128");
    TrunkWeights tw;
    memset(&tw, 0, sizeof(tw));
    if (sample_seed) {
        uint32_t k0 = (uint32_t)*sample_seed, k1 = (uint32_t)(*sample_seed >> 32);
        for (int r = 0; r < 10; ++r) { tw.rk0[r] = k0; tw.rk1[r] = k1; k0 += PHILOX_W0; k1 += PHILOX_W1; }
    }
    tw.w_heads = d_w_heads; tw.b_heads = d_b_heads; tw.n_actions = n_actions; tw.clamp_lo = clamp_lo; tw.clamp_hi = clamp_hi;
    tw.actions = d_actions; tw.value = d_value; tw.probs = d_probs; tw.logp = d_logp; tw.member_rows = member_rows;
    return policy_trunk_launch(h, d_features, (int64_t)n_members * member_rows, d_packed1, d_bias1, d_packed2, d_bias2, hidden2,
                               d_packed3, d_bias3, noise_scale, leaky_slope, d_counter, d_z3, stream, &tw, !sample_seed);
}

int wab_policy_forward_population(WabVec* h, const uint8_t* d_features, int32_t n_members, int64_t member_rows,
                                  const void* d_packed1, const float* d_bias1, const void* d_packed2, const float* d_bias2,
                                  int32_t hidden2, const void* d_packed3, const float* d_bias3, const float* d_w_heads,
                                  const float* d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope, float clamp_lo,
                                  float clamp_hi, uint64_t sample_seed, const uint64_t* d_counter, uint8_t* d_actions,
                                  float* d_value, float* d_probs, float* d_logp, float* d_z3, void* stream) {
    return policy_population_launch("wab_policy_forward_population", h, d_features, n_members, member_rows, d_packed1, d_bias1,
                                    d_packed2, d_bias2, hidden2, d_packed3, d_bias3, d_w_heads, d_b_heads, n_actions, noise_scale,
                                    leaky_slope, clamp_lo, clamp_hi, &sample_seed, d_counter, d_actions, d_value, d_probs, d_logp,
                                    d_z3, stream);
}

int wab_policy_act_population(WabVec* h, const uint8_t* d_features, int32_t n_members, int64_t member_rows,
                              const void* d_packed1, const float* d_bias1, const void* d_packed2, const float* d_bias2,
                              int32_t hidden2, const void* d_packed3, const float* d_bias3, const float* d_w_heads,
                              const float* d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope, float clamp_lo,
                              float clamp_hi, const uint64_t* d_counter, uint8_t* d_actions, float* d_value, float* d_probs,
                              float* d_logp, float* d_z3, void* stream) {
    return policy_population_launch("wab_policy_act_population", h, d_features, n_members, member_rows, d_packed1, d_bias1,
                                    d_packed2, d_bias2, hidden2, d_packed3, d_bias3, d_w_heads, d_b_heads, n_actions, noise_scale,
                                    leaky_slope, clamp_lo, clamp_hi, nullptr, d_counter, d_actions, d_value, d_probs, d_logp,
                                    d_z3, stream);
}

// wab_policy_forward's trunk and tail with the greedy action: the same checks, no sampling seed (MODE 3 reads no round keys)
int wab_policy_act(WabVec* h, const uint8_t* d_features, int64_t n_rows, const void* d_packed1, const float* d_bias1,
                   const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                   const float* d_w_heads, const float* d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                   float clamp_lo, float clamp_hi, const uint64_t* d_counter, uint8_t* d_actions, float* d_value,
                   float* d_probs, float* d_logp, float* d_z3, void* stream) {
    if (!d_w_heads || !d_b_heads || !d_actions) return fail(WAB_E_NULL, "null argument");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_CONFIG, "n_actions must be in [1, 8]");
    TrunkWeights tw;
    memset(&tw, 0, sizeof(tw));
    tw.w_heads = d_w_heads; tw.b_heads = d_b_heads; tw.n_actions = n_actions; tw.clamp_lo = clamp_lo; tw.clamp_hi = clamp_hi;
    tw.actions = d_actions; tw.value = d_value; tw.probs = d_probs; tw.logp = d_logp;
    return policy_trunk_launch(h, d_features, n_rows, d_packed1, d_bias1, d_packed2, d_bias2, hidden2, d_packed3, d_bias3, noise_scale,
                               leaky_slope, d_counter, d_z3, stream, &tw, true);
}

int wab_policy_tail(const float* d_z3, int32_t hidden, const float* d_w_heads, const float* d_b_heads, int64_t n_rows,
                    int32_t n_actions, float leaky_slope, float clamp_lo, float clamp_hi, uint64_t seed,
                    const uint64_t* d_counter, uint8_t* d_actions, float* d_value, float* d_probs, float* d_logp, void* stream) {
    if (!d_z3 || !d_w_heads || !d_b_heads || !d_actions) return fail(WAB_E_NULL, "null argument");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_CONFIG, "n_actions must be in [1, 8]");
    if (hidden != 128) return fail(WAB_E_UNSUPPORTED, "wab_policy_tail is built for the reference's 128-wide trunk (actor_critic.py:65-70)");
    if (n_rows <= 0) return WAB_OK;
    Params P;
    memset(&P, 0, sizeof(P));
    fill_round_keys(P, (uint32_t)seed, (uint32_t)(seed >> 32));
    int dev = 0, n_sm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    const int64_t want = (n_rows + 7) / 8;
    const unsigned grid = (unsigned)(want < (int64_t)n_sm * 8 ? want : (int64_t)n_sm * 8);
    wab_policy_tail_kernel<128><<<grid, 256, 0, (cudaStream_t)stream>>>(
        P, d_z3, d_w_heads, d_b_heads, n_rows, n_actions, leaky_slope, clamp_lo, clamp_hi,
        reinterpret_cast<const unsigned long long*>(d_counter), d_actions, d_value, d_probs, d_logp);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

static int backward_grid(int device) {
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    return n_sm;
}

int64_t wab_policy_backward_scratch_bytes(const WabVec* h) {
    return h ? (int64_t)backward_grid(h->device) * BP_BLOCK * (int64_t)sizeof(float) : 0;
}

// parameters of the reference's Policy with a `dim`-wide input and `n_actions` actions (the flat gradient's length)
static int64_t policy_n_params(int dim, int n_actions) {
    return 128LL * dim + 128 + 150 * 128 + 150 + 128 * 150 + 128 + (int64_t)(n_actions + 1) * 129;
}

int64_t wab_policy_backward_population_scratch_bytes(const WabVec* h, int32_t n_members) {
    return n_members >= 1 && n_members <= 64 ? n_members * wab_policy_backward_scratch_bytes(h) : 0;
}

int64_t wab_policy_population_grad_stride(const WabVec* h, int32_t n_actions) {
    if (!h || n_actions < 1 || n_actions > 8) return 0;
    return (policy_n_params(wab_vec_flat_dim(h), n_actions) + 63) / 64 * 64;
}

// wab_policy_backward and wab_policy_ppo_backward: the checks they share, then the backward kernel (the PPO one when
// `ppo` is given) and the reduction. `d_g_logp` / `d_g_value` are wab_policy_backward's, checked by the caller.
static int policy_backward_launch(const char* who, WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs,
                                  const uint64_t* d_counters, const uint8_t* d_actions, const float* d_g_logp,
                                  const float* d_g_value, const PpoArgs* ppo, const int32_t* d_rows, const int64_t* d_n_rows,
                                  const void* d_packed1, const float* d_bias1, const void* d_packed2, const float* d_bias2,
                                  int32_t hidden2, const void* d_packed3, const float* d_bias3, const void* d_packed2t,
                                  const void* d_packed3t, const float* d_w_heads, const float* d_b_heads, int32_t n_actions,
                                  float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi, void* d_scratch,
                                  int64_t scratch_bytes, float* d_grad, float* d_logp, float* d_value, void* stream,
                                  const PopulationArgs* pop = nullptr, int n_members = 1) {
    if (!h || !d_features || !d_counters || !d_actions || !d_packed1 || !d_bias1 || !d_packed2 ||
        !d_bias2 || !d_packed3 || !d_bias3 || !d_packed2t || !d_packed3t || !d_w_heads || !d_b_heads || !d_scratch || !d_grad)
        return fail(WAB_E_NULL, "null argument");
    if ((d_rows == nullptr) != (d_n_rows == nullptr)) return fail(WAB_E_NULL, "d_rows and d_n_rows go together");
    if (hidden2 != 150) return fail(WAB_E_UNSUPPORTED, std::string(who) + " is built for the reference's trunk 128 -> 150 -> 128 (actor_critic.py:59-61)");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_UNSUPPORTED, std::string(who) + ": at most 8 actions");
    const int dim = wab_vec_flat_dim(h);
    if (dim > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, std::string(who) + ": the input is at most 512 columns wide");
    if (n_steps < 0 || n_envs < 0 || n_steps * n_envs > INT32_MAX) return fail(WAB_E_CONFIG, std::string(who) + ": 0 <= T N < 2^31 rows");
    if (((uintptr_t)d_packed1 & 15u) != 0 || ((uintptr_t)d_packed2 & 15u) != 0 || ((uintptr_t)d_packed3 & 15u) != 0 ||
        ((uintptr_t)d_packed2t & 15u) != 0 || ((uintptr_t)d_packed3t & 15u) != 0 || ((uintptr_t)d_scratch & 15u) != 0 ||
        ((uintptr_t)d_features & 3u) != 0 || ((uintptr_t)d_counters & 7u) != 0 || ((uintptr_t)d_n_rows & 7u) != 0 ||
        ((uintptr_t)d_rows & 3u) != 0 || ((uintptr_t)d_grad & 3u) != 0 || ((uintptr_t)d_g_logp & 3u) != 0 ||
        ((uintptr_t)d_g_value & 3u) != 0 || ((uintptr_t)d_logp & 3u) != 0 || ((uintptr_t)d_value & 3u) != 0 ||
        (ppo && (((uintptr_t)ppo->logp_old & 3u) != 0 || ((uintptr_t)ppo->advantage & 3u) != 0 ||
                 ((uintptr_t)ppo->target & 3u) != 0 || ((uintptr_t)ppo->entropy_out & 3u) != 0)))
        return fail(WAB_E_CONFIG, "the packed weights and d_scratch must be 16-byte aligned, d_counters and d_n_rows 8-byte, "
                                  "d_features, d_rows and the float arrays 4-byte");
    if (scratch_bytes < n_members * wab_policy_backward_scratch_bytes(h))
        return fail(WAB_E_CONFIG, pop ? "d_scratch is smaller than wab_policy_backward_population_scratch_bytes"
                                      : "d_scratch is smaller than wab_policy_backward_scratch_bytes");
    DeviceGuard guard(h->device);
    static bool attr_set[3][64] = {{false}};
    const int kind = pop ? 2 : ppo ? 1 : 0;
    if (h->device < 64 && !attr_set[kind][h->device]) {
        if (pop) WAB_CUDA(cudaFuncSetAttribute(wab_policy_ppo_bwd_population_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_SMEM_TOTAL));
        else if (ppo) WAB_CUDA(cudaFuncSetAttribute(wab_policy_ppo_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_SMEM_TOTAL));
        else WAB_CUDA(cudaFuncSetAttribute(wab_policy_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_SMEM_TOTAL));
        attr_set[kind][h->device] = true;
    }
    BackwardArgs B;
    memset(&B, 0, sizeof(B));
    B.features = d_features; B.n_envs = n_envs > 0 ? n_envs : 1; B.n_rows = n_steps * n_envs;
    B.counters = reinterpret_cast<const unsigned long long*>(d_counters);
    B.actions = d_actions; B.g_logp = d_g_logp; B.g_value = d_g_value;
    B.rows = d_rows; B.d_count = reinterpret_cast<const long long*>(d_n_rows);
    B.w1 = reinterpret_cast<const uint4*>(d_packed1); B.b1 = d_bias1; B.w2 = reinterpret_cast<const uint4*>(d_packed2); B.b2 = d_bias2;
    B.w3 = reinterpret_cast<const uint4*>(d_packed3); B.b3 = d_bias3;
    B.w2t = reinterpret_cast<const uint4*>(d_packed2t); B.w3t = reinterpret_cast<const uint4*>(d_packed3t);
    B.w_heads = d_w_heads; B.b_heads = d_b_heads; B.n_actions = n_actions; B.noise_scale = noise_scale; B.slope = leaky_slope;
    B.clamp_lo = clamp_lo; B.clamp_hi = clamp_hi; B.scratch = reinterpret_cast<float*>(d_scratch);
    B.logp_out = d_logp; B.value_out = d_value;
    const int grid = backward_grid(h->device);
    const int64_t total = policy_n_params(dim, n_actions);
    if (pop) {
        PopulationArgs G = *pop;
        G.n_cta = grid;
        wab_policy_ppo_bwd_population_kernel<<<grid * n_members, 256, BW_SMEM_TOTAL, (cudaStream_t)stream>>>(
            h->P, (int)h->cfg.food_obs_scale + 1, B, *ppo, G);
        WAB_CUDA(cudaGetLastError());
        wab_policy_bwd_reduce_population_kernel<float><<<dim3((unsigned)((total + 255) / 256), (unsigned)n_members), 256, 0, (cudaStream_t)stream>>>(
            reinterpret_cast<const float*>(d_scratch), grid, dim, n_actions, (total + 63) / 64 * 64, d_grad);
        WAB_CUDA(cudaGetLastError());
        return WAB_OK;
    }
    if (ppo) wab_policy_ppo_bwd_kernel<<<grid, 256, BW_SMEM_TOTAL, (cudaStream_t)stream>>>(h->P, (int)h->cfg.food_obs_scale + 1, B, *ppo);
    else wab_policy_bwd_kernel<<<grid, 256, BW_SMEM_TOTAL, (cudaStream_t)stream>>>(h->P, (int)h->cfg.food_obs_scale + 1, B);
    WAB_CUDA(cudaGetLastError());
    wab_policy_bwd_reduce_kernel<float><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(d_scratch), grid, dim, n_actions, d_grad);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_policy_backward(WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs, const uint64_t* d_counters,
                        const uint8_t* d_actions, const float* d_g_logp, const float* d_g_value, const int32_t* d_rows,
                        const int64_t* d_n_rows, const void* d_packed1, const float* d_bias1, const void* d_packed2,
                        const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                        const void* d_packed2t, const void* d_packed3t, const float* d_w_heads, const float* d_b_heads,
                        int32_t n_actions, float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi,
                        void* d_scratch, int64_t scratch_bytes, float* d_grad, float* d_logp, float* d_value, void* stream) {
    if (!d_g_logp || !d_g_value) return fail(WAB_E_NULL, "null argument");
    return policy_backward_launch("wab_policy_backward", h, d_features, n_steps, n_envs, d_counters, d_actions, d_g_logp,
                                  d_g_value, nullptr, d_rows, d_n_rows, d_packed1, d_bias1, d_packed2, d_bias2, hidden2,
                                  d_packed3, d_bias3, d_packed2t, d_packed3t, d_w_heads, d_b_heads, n_actions, noise_scale,
                                  leaky_slope, clamp_lo, clamp_hi, d_scratch, scratch_bytes, d_grad, d_logp, d_value, stream);
}

int wab_policy_ppo_backward(WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs, const uint64_t* d_counters,
                            const uint8_t* d_actions, const float* d_logp_old, const float* d_advantage, const float* d_target,
                            const int32_t* d_rows, const int64_t* d_n_rows, const void* d_packed1, const float* d_bias1,
                            const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3,
                            const float* d_bias3, const void* d_packed2t, const void* d_packed3t, const float* d_w_heads,
                            const float* d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope, float clamp_lo,
                            float clamp_hi, float clip_eps, float policy_weight, float value_weight, float entropy_weight,
                            void* d_scratch, int64_t scratch_bytes, float* d_grad, float* d_logp, float* d_value,
                            float* d_entropy, void* stream) {
    if (!d_logp_old || !d_advantage || !d_target) return fail(WAB_E_NULL, "null argument");
    if (!(clip_eps > 0.f)) return fail(WAB_E_CONFIG, "wab_policy_ppo_backward: clip_eps must be > 0 (+inf disables clipping)");
    if (!std::isfinite(policy_weight) || !std::isfinite(value_weight) || !std::isfinite(entropy_weight))
        return fail(WAB_E_CONFIG, "wab_policy_ppo_backward: the loss weights must be finite");
    PpoArgs Q;
    memset(&Q, 0, sizeof(Q));
    Q.logp_old = d_logp_old; Q.advantage = d_advantage; Q.target = d_target;
    Q.clip_eps = clip_eps; Q.w_policy = policy_weight; Q.w_value = value_weight; Q.w_entropy = entropy_weight;
    Q.entropy_out = d_entropy;
    return policy_backward_launch("wab_policy_ppo_backward", h, d_features, n_steps, n_envs, d_counters, d_actions, nullptr,
                                  nullptr, &Q, d_rows, d_n_rows, d_packed1, d_bias1, d_packed2, d_bias2, hidden2, d_packed3,
                                  d_bias3, d_packed2t, d_packed3t, d_w_heads, d_b_heads, n_actions, noise_scale, leaky_slope,
                                  clamp_lo, clamp_hi, d_scratch, scratch_bytes, d_grad, d_logp, d_value, stream);
}

int wab_policy_ppo_backward_population(WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs, int32_t n_members,
                                       const uint64_t* d_counters, const uint8_t* d_actions, const float* d_logp_old,
                                       const float* d_advantage, const float* d_target, const int32_t* d_rows, int64_t list_len,
                                       const int64_t* d_counts, const void* d_packed1, const float* d_bias1,
                                       const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3,
                                       const float* d_bias3, const void* d_packed2t, const void* d_packed3t,
                                       const float* d_w_heads, const float* d_b_heads, int32_t n_actions, float noise_scale,
                                       float leaky_slope, float clamp_lo, float clamp_hi, const float* h_coefs,
                                       void* d_scratch, int64_t scratch_bytes, float* d_grad, float* d_logp, float* d_value,
                                       float* d_entropy, void* stream) {
    if (!d_logp_old || !d_advantage || !d_target || !d_rows || !d_counts || !h_coefs) return fail(WAB_E_NULL, "null argument");
    if (n_members < 1 || n_members > 64) return fail(WAB_E_CONFIG, "wab_policy_ppo_backward_population: 1 <= n_members <= 64");
    if (n_envs % n_members != 0 || (n_envs / n_members) % TC_TILE_M != 0 || n_envs == 0)
        return fail(WAB_E_CONFIG, "wab_policy_ppo_backward_population: n_envs / n_members must be a positive multiple of 128");
    if (list_len < 0) return fail(WAB_E_CONFIG, "wab_policy_ppo_backward_population: list_len must be >= 0");
    PopulationArgs G;
    memset(&G, 0, sizeof(G));
    for (int m = 0; m < n_members; ++m) {
        const float* c = h_coefs + 4 * m;
        if (!(c[0] > 0.f)) return fail(WAB_E_CONFIG, "wab_policy_ppo_backward_population: clip_eps must be > 0 (+inf disables clipping)");
        if (!std::isfinite(c[1]) || !std::isfinite(c[2]) || !std::isfinite(c[3]))
            return fail(WAB_E_CONFIG, "wab_policy_ppo_backward_population: the loss weights must be finite");
        for (int k = 0; k < 4; ++k) G.coef[m][k] = c[k];
    }
    G.member_envs = n_envs / n_members; G.list_len = list_len; G.rows = d_rows;
    G.counts = reinterpret_cast<const long long*>(d_counts);
    PpoArgs Q;
    memset(&Q, 0, sizeof(Q));
    Q.logp_old = d_logp_old; Q.advantage = d_advantage; Q.target = d_target; Q.entropy_out = d_entropy;
    return policy_backward_launch("wab_policy_ppo_backward_population", h, d_features, n_steps, n_envs, d_counters, d_actions,
                                  nullptr, nullptr, &Q, d_rows, d_counts, d_packed1, d_bias1, d_packed2, d_bias2, hidden2,
                                  d_packed3, d_bias3, d_packed2t, d_packed3t, d_w_heads, d_b_heads, n_actions, noise_scale,
                                  leaky_slope, clamp_lo, clamp_hi, d_scratch, scratch_bytes, d_grad, d_logp, d_value, stream,
                                  &G, n_members);
}

// wab_policy_evaluate and wab_policy_backward_logits: the checks they share, then the list kernel (the evaluation when
// `d_logits` is given, else the logits backward followed by the reduction). The per-kind arrays are checked by the callers.
static int policy_list_launch(const char* who, WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs,
                              const uint64_t* d_counters, const int32_t* d_rows, int64_t n_rows, const float* d_g_logits,
                              const float* d_g_value, const void* d_packed1, const float* d_bias1, const void* d_packed2,
                              const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                              const void* d_packed2t, const void* d_packed3t, const float* d_w_heads, const float* d_b_heads,
                              int32_t n_actions, float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi,
                              void* d_scratch, int64_t scratch_bytes, float* d_grad, float* d_logits, float* d_value,
                              void* stream) {
    if (!h || !d_features || !d_counters || !d_packed1 || !d_bias1 || !d_packed2 || !d_bias2 || !d_packed3 || !d_bias3 ||
        !d_w_heads || !d_b_heads || !d_scratch)
        return fail(WAB_E_NULL, "null argument");
    if (hidden2 != 150) return fail(WAB_E_UNSUPPORTED, std::string(who) + " is built for the reference's trunk 128 -> 150 -> 128 (actor_critic.py:59-61)");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_UNSUPPORTED, std::string(who) + ": at most 8 actions");
    const int dim = wab_vec_flat_dim(h);
    if (dim > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, std::string(who) + ": the input is at most 512 columns wide");
    if (n_steps < 0 || n_envs < 0 || n_steps * n_envs > INT32_MAX) return fail(WAB_E_CONFIG, std::string(who) + ": 0 <= T N < 2^31 rows");
    if (n_rows < 0) return fail(WAB_E_CONFIG, std::string(who) + ": n_rows must be >= 0");
    if (!(noise_scale >= 0.f) || !std::isfinite(noise_scale)) return fail(WAB_E_CONFIG, std::string(who) + ": noise_scale must be finite and >= 0");
    if (((uintptr_t)d_packed1 & 15u) != 0 || ((uintptr_t)d_packed2 & 15u) != 0 || ((uintptr_t)d_packed3 & 15u) != 0 ||
        ((uintptr_t)d_packed2t & 15u) != 0 || ((uintptr_t)d_packed3t & 15u) != 0 || ((uintptr_t)d_scratch & 15u) != 0 ||
        ((uintptr_t)d_features & 3u) != 0 || ((uintptr_t)d_counters & 7u) != 0 || ((uintptr_t)d_rows & 3u) != 0 ||
        ((uintptr_t)d_grad & 3u) != 0 || ((uintptr_t)d_g_logits & 3u) != 0 || ((uintptr_t)d_g_value & 3u) != 0 ||
        ((uintptr_t)d_logits & 3u) != 0 || ((uintptr_t)d_value & 3u) != 0)
        return fail(WAB_E_CONFIG, "the packed weights and d_scratch must be 16-byte aligned, d_counters 8-byte, "
                                  "d_features, d_rows and the float arrays 4-byte");
    if (scratch_bytes < wab_policy_backward_scratch_bytes(h)) return fail(WAB_E_CONFIG, "d_scratch is smaller than wab_policy_backward_scratch_bytes");
    const bool eval = d_logits != nullptr;
    DeviceGuard guard(h->device);
    static bool attr_set[2][64] = {{false}};
    if (h->device < 64 && !attr_set[eval ? 1 : 0][h->device]) {
        if (eval) WAB_CUDA(cudaFuncSetAttribute(wab_policy_eval_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_SMEM_TOTAL));
        else WAB_CUDA(cudaFuncSetAttribute(wab_policy_logits_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_SMEM_TOTAL));
        attr_set[eval ? 1 : 0][h->device] = true;
    }
    BackwardArgs B;
    memset(&B, 0, sizeof(B));
    B.features = d_features; B.n_envs = n_envs > 0 ? n_envs : 1; B.n_rows = n_steps * n_envs;
    B.counters = reinterpret_cast<const unsigned long long*>(d_counters);
    B.rows = d_rows;
    B.w1 = reinterpret_cast<const uint4*>(d_packed1); B.b1 = d_bias1; B.w2 = reinterpret_cast<const uint4*>(d_packed2); B.b2 = d_bias2;
    B.w3 = reinterpret_cast<const uint4*>(d_packed3); B.b3 = d_bias3;
    B.w2t = reinterpret_cast<const uint4*>(d_packed2t); B.w3t = reinterpret_cast<const uint4*>(d_packed3t);
    B.w_heads = d_w_heads; B.b_heads = d_b_heads; B.n_actions = n_actions; B.noise_scale = noise_scale; B.slope = leaky_slope;
    B.clamp_lo = clamp_lo; B.clamp_hi = clamp_hi; B.scratch = reinterpret_cast<float*>(d_scratch);
    ListArgs L;
    memset(&L, 0, sizeof(L));
    L.n_list = n_rows; L.g_logits = d_g_logits; L.g_value = d_g_value; L.logits_out = d_logits; L.value_out = d_value;
    const int grid = backward_grid(h->device);
    if (eval) {
        wab_policy_eval_kernel<<<grid, 256, BW_SMEM_TOTAL, (cudaStream_t)stream>>>(h->P, (int)h->cfg.food_obs_scale + 1, B, L);
        WAB_CUDA(cudaGetLastError());
        return WAB_OK;
    }
    wab_policy_logits_bwd_kernel<<<grid, 256, BW_SMEM_TOTAL, (cudaStream_t)stream>>>(h->P, (int)h->cfg.food_obs_scale + 1, B, L);
    WAB_CUDA(cudaGetLastError());
    const int64_t total = policy_n_params(dim, n_actions);
    wab_policy_bwd_reduce_kernel<float><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(d_scratch), grid, dim, n_actions, d_grad);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_policy_evaluate(WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs, const uint64_t* d_counters,
                        const int32_t* d_rows, int64_t n_rows, const void* d_packed1, const float* d_bias1,
                        const void* d_packed2, const float* d_bias2, int32_t hidden2, const void* d_packed3,
                        const float* d_bias3, const float* d_w_heads, const float* d_b_heads, int32_t n_actions,
                        float noise_scale, float leaky_slope, float clamp_lo, float clamp_hi, void* d_scratch,
                        int64_t scratch_bytes, float* d_logits, float* d_value, void* stream) {
    if (!d_logits || !d_value) return fail(WAB_E_NULL, "null argument");
    // the evaluation runs no step 3: the transposed weights are never read, the forward's stand in for the checks
    return policy_list_launch("wab_policy_evaluate", h, d_features, n_steps, n_envs, d_counters, d_rows, n_rows, nullptr,
                              nullptr, d_packed1, d_bias1, d_packed2, d_bias2, hidden2, d_packed3, d_bias3, d_packed2,
                              d_packed3, d_w_heads, d_b_heads, n_actions, noise_scale, leaky_slope, clamp_lo, clamp_hi,
                              d_scratch, scratch_bytes, nullptr, d_logits, d_value, stream);
}

int wab_policy_backward_logits(WabVec* h, const uint8_t* d_features, int64_t n_steps, int64_t n_envs,
                               const uint64_t* d_counters, const int32_t* d_rows, int64_t n_rows, const float* d_g_logits,
                               const float* d_g_value, const void* d_packed1, const float* d_bias1, const void* d_packed2,
                               const float* d_bias2, int32_t hidden2, const void* d_packed3, const float* d_bias3,
                               const void* d_packed2t, const void* d_packed3t, const float* d_w_heads,
                               const float* d_b_heads, int32_t n_actions, float noise_scale, float leaky_slope,
                               float clamp_lo, float clamp_hi, void* d_scratch, int64_t scratch_bytes, float* d_grad,
                               void* stream) {
    if (!d_g_logits || !d_g_value || !d_packed2t || !d_packed3t || !d_grad) return fail(WAB_E_NULL, "null argument");
    return policy_list_launch("wab_policy_backward_logits", h, d_features, n_steps, n_envs, d_counters, d_rows, n_rows,
                              d_g_logits, d_g_value, d_packed1, d_bias1, d_packed2, d_bias2, hidden2, d_packed3, d_bias3,
                              d_packed2t, d_packed3t, d_w_heads, d_b_heads, n_actions, noise_scale, leaky_slope, clamp_lo,
                              clamp_hi, d_scratch, scratch_bytes, d_grad, nullptr, nullptr, stream);
}

int wab_policy_backward_grad_f64(WabVec* h, const void* d_scratch, int64_t scratch_bytes, int32_t n_actions, double* d_grad64,
                                 void* stream) {
    if (!h || !d_scratch || !d_grad64) return fail(WAB_E_NULL, "null argument");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_UNSUPPORTED, "wab_policy_backward_grad_f64: at most 8 actions");
    const int dim = wab_vec_flat_dim(h);
    if (dim > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, "wab_policy_backward_grad_f64: the input is at most 512 columns wide");
    if (((uintptr_t)d_scratch & 15u) != 0 || ((uintptr_t)d_grad64 & 7u) != 0)
        return fail(WAB_E_CONFIG, "d_scratch must be 16-byte aligned, d_grad64 8-byte");
    if (scratch_bytes < wab_policy_backward_scratch_bytes(h)) return fail(WAB_E_CONFIG, "d_scratch is smaller than wab_policy_backward_scratch_bytes");
    DeviceGuard guard(h->device);
    const int64_t total = policy_n_params(dim, n_actions);
    wab_policy_bwd_reduce_kernel<double><<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(d_scratch), backward_grid(h->device), dim, n_actions, d_grad64);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_policy_backward_population_grad_f64(WabVec* h, const void* d_scratch, int64_t scratch_bytes, int32_t n_members,
                                            int32_t n_actions, double* d_grad64, void* stream) {
    if (!h || !d_scratch || !d_grad64) return fail(WAB_E_NULL, "null argument");
    if (n_members < 1 || n_members > 64) return fail(WAB_E_CONFIG, "wab_policy_backward_population_grad_f64: 1 <= n_members <= 64");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_UNSUPPORTED, "wab_policy_backward_population_grad_f64: at most 8 actions");
    const int dim = wab_vec_flat_dim(h);
    if (dim > TC_CHUNKS * TC_KC) return fail(WAB_E_UNSUPPORTED, "wab_policy_backward_population_grad_f64: the input is at most 512 columns wide");
    if (((uintptr_t)d_scratch & 15u) != 0 || ((uintptr_t)d_grad64 & 7u) != 0)
        return fail(WAB_E_CONFIG, "d_scratch must be 16-byte aligned, d_grad64 8-byte");
    if (scratch_bytes < n_members * wab_policy_backward_scratch_bytes(h))
        return fail(WAB_E_CONFIG, "d_scratch is smaller than wab_policy_backward_population_scratch_bytes");
    DeviceGuard guard(h->device);
    const int64_t stride = wab_policy_population_grad_stride(h, n_actions);
    wab_policy_bwd_reduce_population_kernel<double><<<dim3((unsigned)((stride + 255) / 256), (unsigned)n_members), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(d_scratch), backward_grid(h->device), dim, n_actions, stride, d_grad64);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_policy_grad_sum_ranks(const double* d_rank_grads, int32_t n_ranks, int64_t n, float* d_grad, void* stream) {
    if (!d_rank_grads || !d_grad) return fail(WAB_E_NULL, "null argument");
    if (n_ranks < 1) return fail(WAB_E_CONFIG, "wab_policy_grad_sum_ranks: n_ranks must be >= 1");
    if (n < 0) return fail(WAB_E_CONFIG, "wab_policy_grad_sum_ranks: n must be >= 0");
    if (((uintptr_t)d_rank_grads & 7u) != 0 || ((uintptr_t)d_grad & 3u) != 0)
        return fail(WAB_E_CONFIG, "d_rank_grads must be 8-byte aligned, d_grad 4-byte");
    if (n == 0) return WAB_OK;
    wab_policy_grad_sum_ranks_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_rank_grads, n_ranks, n, d_grad);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_sample_categorical(const void* d_probs, int32_t probs_bf16, int64_t n, int32_t n_actions, uint64_t seed,
                           const uint64_t* d_counter, uint8_t* d_actions, void* stream) {
    if (!d_probs || !d_actions) return fail(WAB_E_NULL, "null argument");
    if (n_actions < 1 || n_actions > 8) return fail(WAB_E_CONFIG, "n_actions must be in [1, 8]");
    if (n <= 0) return WAB_OK;
    Params P;
    memset(&P, 0, sizeof(P));
    fill_round_keys(P, (uint32_t)seed, (uint32_t)(seed >> 32));
    const unsigned grid = (unsigned)((n + 255) / 256);
    const unsigned long long* ctr = reinterpret_cast<const unsigned long long*>(d_counter);
    if (probs_bf16) wab_sample_kernel<1><<<grid, 256, 0, (cudaStream_t)stream>>>(P, d_probs, n, n_actions, ctr, d_actions);
    else wab_sample_kernel<0><<<grid, 256, 0, (cudaStream_t)stream>>>(P, d_probs, n, n_actions, ctr, d_actions);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_philox_device(const uint32_t* d_ctr, uint32_t key0, uint32_t key1, int64_t n, uint32_t* d_out, void* stream) {
    if (!d_ctr || !d_out) return fail(WAB_E_NULL, "null argument");
    if (n <= 0) return WAB_OK;
    Params P;
    memset(&P, 0, sizeof(P));
    fill_round_keys(P, key0, key1);
    wab_philox_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(P, d_ctr, n, d_out);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

}  // extern "C"

#include "wab_state.cuh"
#include "wab2_kernels.cuh"
