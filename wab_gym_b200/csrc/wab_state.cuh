// wab_state.cuh — save / validate / load of per-env state records and their C ABI (included by wab_kernels.cu).
//
// The record layout is documented in include/wab_b200.h (WAB_STATE_FORMAT). The slab is struct-of-arrays ([N] columns,
// [cap][N] slot columns), a record is one env's row: both kernels transpose through shared memory, 32 records per CTA,
// so that the column accesses of consecutive threads hit consecutive envs and the record side moves as 16-byte words.
// Shared memory holds record e at word e * SW with SW = record words | 1 (odd: the per-env column pass is free of bank
// conflicts). Only live wolf, log and history slots are read or written; dead slots of a record are zero.
#pragma once

namespace {

constexpr int kStateEnvs = 32;       // records per CTA
constexpr int kStateThreads = 256;

// word offsets of the fixed part (byte offset / 4, include/wab_b200.h)
enum : int {
    RW_FORMAT = 0, RW_FLAGS = 1, RW_FP = 2, RW_ENV_ID = 4, RW_EPISODE = 6, RW_TURN = 7, RW_X = 8, RW_Y = 9, RW_ROLE = 10,
    RW_STATUS = 11, RW_FOOD_I = 12, RW_NW = 13, RW_FOOD_F = 14, RW_BKEY = 16, RW_NLOG = 18, RW_WINDOW = 20, RW_HEAD = 24
};

struct RecGeo {
    int32_t wolves, logcell, logcnt_byte, hist;   // word offsets (logcnt: byte offset)
    int32_t words, sw;                             // record words, shared-memory stride in words
    int32_t wolf_cap, log_cap, hist_len;           // hist_len 0 without ego
};

RecGeo rec_geo(const WabVec* h) {
    RecGeo g;
    g.wolf_cap = h->cfg.wolf_cap; g.log_cap = h->cfg.log_cap; g.hist_len = h->st.hist ? h->st.hist_len : 0;
    g.wolves = RW_HEAD;
    g.logcell = g.wolves + g.wolf_cap;
    g.logcnt_byte = 4 * (g.logcell + g.log_cap);
    g.hist = (g.logcnt_byte + g.log_cap + 3) / 4;
    g.words = (g.hist + g.hist_len + 3) & ~3;      // 16-byte records
    g.sw = g.words | 1;
    return g;
}

__device__ __forceinline__ uint64_t rec_u64(const uint32_t* r, int w) { return (uint64_t)r[w] | ((uint64_t)r[w + 1] << 32); }

// gather: slab columns of slots[r] (or r) -> records
__global__ void __launch_bounds__(kStateThreads) wab_save_state_kernel(const __grid_constant__ Params P, const StatePtrs st,
                                                                       const RecGeo g, uint64_t fp, int f64,
                                                                       const int32_t* __restrict__ slots, int64_t n_rec,
                                                                       uint4* __restrict__ out) {
    extern __shared__ uint32_t srec[];
    __shared__ int64_t s_slot[kStateEnvs];
    __shared__ int32_t s_nw[kStateEnvs], s_nlog[kStateEnvs], s_hist_hi[kStateEnvs];
    const int64_t r0 = (int64_t)blockIdx.x * kStateEnvs, n = st.n;
    const int nb = (int)(n_rec - r0 < kStateEnvs ? n_rec - r0 : kStateEnvs);
    for (int i = threadIdx.x; i < nb * g.sw; i += blockDim.x) srec[i] = 0u;
    __syncthreads();
    if ((int)threadIdx.x < nb) {
        const int e = threadIdx.x;
        const int64_t idx = slots ? (int64_t)slots[r0 + e] : r0 + e;
        uint32_t* r = srec + e * g.sw;
        const uint32_t pos = st.pos[idx], misc = st.misc[idx], nl = st.nlog[idx];
        const uint32_t nw = ((misc >> 11) & 15u) | (((nl >> 9) & 7u) << 4), nlog = nl & 0xFFu, turn = misc >> 16;
        const uint64_t env_id = global_env_id(P, idx);
        r[RW_FORMAT] = WAB_STATE_FORMAT; r[RW_FLAGS] = (nl >> 8) & 1u;
        r[RW_FP] = (uint32_t)fp; r[RW_FP + 1] = (uint32_t)(fp >> 32);
        r[RW_ENV_ID] = (uint32_t)env_id; r[RW_ENV_ID + 1] = (uint32_t)(env_id >> 32);
        r[RW_EPISODE] = st.episode[idx]; r[RW_TURN] = turn;
        r[RW_X] = (uint32_t)unpack_x(pos); r[RW_Y] = (uint32_t)unpack_y(pos);
        r[RW_ROLE] = (misc >> 8) & 1u; r[RW_STATUS] = (misc >> 9) & 3u;
        r[RW_NW] = nw; r[RW_NLOG] = nlog;
        if (f64) {
            const uint64_t fb = (uint64_t)__double_as_longlong(st.food[idx]);
            r[RW_FOOD_F] = (uint32_t)fb; r[RW_FOOD_F + 1] = (uint32_t)(fb >> 32);
        } else {
            r[RW_FOOD_I] = misc & 0xFFu;
        }
        const uint2 bk = st.bkey[idx];
        r[RW_BKEY] = bk.x; r[RW_BKEY + 1] = bk.y;
        const uint4 m = st.bush[idx];
        r[RW_WINDOW] = m.x; r[RW_WINDOW + 1] = m.y; r[RW_WINDOW + 2] = m.z; r[RW_WINDOW + 3] = m.w;
        s_slot[e] = idx; s_nw[e] = (int32_t)nw; s_nlog[e] = (int32_t)nlog;
        s_hist_hi[e] = (int32_t)(turn < (uint32_t)g.hist_len ? turn : (uint32_t)g.hist_len - 1u);   // hist[1 .. hi] are live
    }
    __syncthreads();
    // slot columns: consecutive threads read consecutive envs of one column
    for (int i = threadIdx.x; i < g.wolf_cap * nb; i += blockDim.x) {
        const int k = i / nb, e = i - k * nb;
        if (k < s_nw[e]) srec[e * g.sw + g.wolves + k] = st.wolves[(int64_t)k * n + s_slot[e]];
    }
    for (int i = threadIdx.x; i < g.log_cap * nb; i += blockDim.x) {
        const int k = i / nb, e = i - k * nb;
        if (k < s_nlog[e]) {
            srec[e * g.sw + g.logcell + k] = st.logcell[(int64_t)k * n + s_slot[e]];
            reinterpret_cast<uint8_t*>(srec + e * g.sw)[g.logcnt_byte + k] = st.logcnt[(int64_t)k * n + s_slot[e]];
        }
    }
    for (int i = threadIdx.x; i < g.hist_len * nb; i += blockDim.x) {
        const int t = i / nb, e = i - t * nb;
        if (t >= 1 && t <= s_hist_hi[e]) srec[e * g.sw + g.hist + t] = st.hist[(int64_t)t * n + s_slot[e]];
    }
    __syncthreads();
    const int q = g.words / 4;                     // 16-byte words per record
    uint4* dst = out + r0 * q;
    for (int c = threadIdx.x; c < nb * q; c += blockDim.x) {
        const int e = c / q, w = (c - e * q) * 4;
        const uint32_t* s = srec + e * g.sw + w;
        dst[c] = make_uint4(s[0], s[1], s[2], s[3]);
    }
}

// Validation pass: *rejected += number of records that must not be loaded. A record passes only if everything the
// kernels index with (slot, n_wolves, n_log) is inside its cap and every field is a value the kernels maintain.
__global__ void __launch_bounds__(kStateThreads) wab_validate_state_kernel(const __grid_constant__ Params P, const RecGeo g,
                                                                           uint64_t fp, int f64, int64_t n_envs,
                                                                           const uint32_t* __restrict__ recs,
                                                                           const int32_t* __restrict__ slots, int64_t n_rec,
                                                                           int32_t* __restrict__ rejected) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool bad = false;
    if (r < n_rec) {
        const uint32_t* h = recs + r * g.words;
        const int64_t slot = slots ? (int64_t)slots[r] : r;
        bad = h[RW_FORMAT] != WAB_STATE_FORMAT || rec_u64(h, RW_FP) != fp || slot < 0 || slot >= n_envs ||
              h[RW_FLAGS] > 1u || h[RW_TURN] > 0xFFFFu || h[RW_ROLE] > 1u || h[RW_STATUS] > 2u ||
              h[RW_NW] > (uint32_t)g.wolf_cap || h[RW_NLOG] > (uint32_t)g.log_cap ||
              (!f64 && h[RW_FOOD_I] > (uint32_t)P.food_int_max);
    }
    const unsigned nbad = __popc(__ballot_sync(0xFFFFFFFFu, bad));
    if ((threadIdx.x & 31) == 0 && nbad) atomicAdd(rejected, (int32_t)nbad);
}

// scatter: records -> slab columns of slots[r] (or r); the log's Bloom signature and the "eaten empty" flag are rebuilt.
// Reads *rejected first and writes nothing when the validation pass refused any record.
__global__ void __launch_bounds__(kStateThreads) wab_load_state_kernel(const __grid_constant__ Params P, const StatePtrs st,
                                                                       const RecGeo g, int f64,
                                                                       const uint4* __restrict__ recs,
                                                                       const int32_t* __restrict__ slots, int64_t n_rec,
                                                                       const int32_t* __restrict__ rejected) {
    if (*rejected != 0) return;
    extern __shared__ uint32_t srec[];
    __shared__ int64_t s_slot[kStateEnvs];
    __shared__ int32_t s_nw[kStateEnvs], s_nlog[kStateEnvs], s_hist_hi[kStateEnvs];
    const int64_t r0 = (int64_t)blockIdx.x * kStateEnvs, n = st.n;
    const int nb = (int)(n_rec - r0 < kStateEnvs ? n_rec - r0 : kStateEnvs);
    const int q = g.words / 4;
    const uint4* src = recs + r0 * q;
    for (int c = threadIdx.x; c < nb * q; c += blockDim.x) {
        const int e = c / q, w = (c - e * q) * 4;
        const uint4 v = src[c];
        uint32_t* d = srec + e * g.sw + w;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    __syncthreads();
    if ((int)threadIdx.x < nb) {
        const int e = threadIdx.x;
        const int64_t idx = slots ? (int64_t)slots[r0 + e] : r0 + e;
        const uint32_t* r = srec + e * g.sw;
        const uint32_t nw = r[RW_NW], nlog = r[RW_NLOG], turn = r[RW_TURN], stale = r[RW_FLAGS] & 1u;
        const uint32_t bka = r[RW_BKEY], bkb = r[RW_BKEY + 1];
        const uint8_t* cnt = reinterpret_cast<const uint8_t*>(r) + g.logcnt_byte;
        uint32_t logsig = 0u, dep = 0u;
        for (uint32_t l = 0; l < nlog; ++l) {
            const uint32_t cell = r[g.logcell + l];
            logsig |= cell_sig(cell);
            if (!dep) {
                const int32_t x = unpack_x(cell), y = unpack_y(cell);
                const uint32_t word = bush_word_rare(pack_xy(x >> 1, y >> 1) ^ bka, bkb, P.rk2[0], bush_lane(x, y));
                dep = alive_after(P, word, (uint32_t)cnt[l]) ? 0u : 1u;
            }
        }
        const uint32_t food_i = f64 ? ((uint32_t)P.food_int_start & 0xFFu) : r[RW_FOOD_I];
        st.pos[idx] = pack_xy((int32_t)r[RW_X], (int32_t)r[RW_Y]);
        st.misc[idx] = food_i | (r[RW_ROLE] << 8) | (r[RW_STATUS] << 9) | ((nw & 15u) << 11) | (dep << 15) | (turn << 16);
        st.nlog[idx] = (uint16_t)(nlog | (stale << 8) | ((nw >> 4) << 9));
        st.logsig[idx] = logsig;
        st.episode[idx] = r[RW_EPISODE];
        st.bkey[idx] = make_uint2(bka, bkb);
        if (f64) st.food[idx] = __longlong_as_double((long long)rec_u64(r, RW_FOOD_F));
        st.bush[idx] = make_uint4(r[RW_WINDOW], r[RW_WINDOW + 1], r[RW_WINDOW + 2], r[RW_WINDOW + 3]);
        s_slot[e] = idx; s_nw[e] = (int32_t)nw; s_nlog[e] = (int32_t)nlog;
        s_hist_hi[e] = (int32_t)(turn < (uint32_t)g.hist_len ? turn : (uint32_t)g.hist_len - 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < g.wolf_cap * nb; i += blockDim.x) {
        const int k = i / nb, e = i - k * nb;
        if (k < s_nw[e]) st.wolves[(int64_t)k * n + s_slot[e]] = srec[e * g.sw + g.wolves + k];
    }
    for (int i = threadIdx.x; i < g.log_cap * nb; i += blockDim.x) {
        const int k = i / nb, e = i - k * nb;
        if (k < s_nlog[e]) {
            st.logcell[(int64_t)k * n + s_slot[e]] = srec[e * g.sw + g.logcell + k];
            st.logcnt[(int64_t)k * n + s_slot[e]] = reinterpret_cast<const uint8_t*>(srec + e * g.sw)[g.logcnt_byte + k];
        }
    }
    for (int i = threadIdx.x; i < g.hist_len * nb; i += blockDim.x) {
        const int t = i / nb, e = i - t * nb;
        if (t >= 1 && t <= s_hist_hi[e]) st.hist[(int64_t)t * n + s_slot[e]] = srec[e * g.sw + g.hist + t];
    }
}

uint64_t state_fingerprint(const WabVec* h) { return fp_mix(h->fp_config, h->st.hist ? 1u : 0u); }

// records of up to 32 x 5.7 KB (wolf_cap 64, log_cap 255, a 1,024-turn history) need the opt-in shared-memory size
int state_smem(const void* kern, const RecGeo& g, size_t& smem) {
    smem = sizeof(uint32_t) * (size_t)kStateEnvs * (size_t)g.sw;
    if (smem > 48 * 1024) WAB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return WAB_OK;
}

}  // namespace

extern "C" {

int64_t wab_vec_state_record_bytes(const WabVec* h) { return h ? 4 * (int64_t)rec_geo(h).words : 0; }

int wab_vec_state_fingerprint(const WabVec* h, uint64_t* out) {
    if (!h || !out) return fail(WAB_E_NULL, "null argument");
    *out = state_fingerprint(h);
    return WAB_OK;
}

int wab_vec_save_state(WabVec* h, const int32_t* d_slots, int64_t n, void* d_records, void* stream) {
    if (!h || !d_records) return fail(WAB_E_NULL, "null argument");
    if (int rc = check_ptr_align(d_records, "d_records")) return rc;
    if (n < 0 || (!d_slots && n != h->n)) return fail(WAB_E_CONFIG, "without d_slots, n must be the number of envs");
    if (n == 0) return WAB_OK;
    DeviceGuard guard(h->device);
    const RecGeo g = rec_geo(h);
    size_t smem;
    if (int rc = state_smem((const void*)wab_save_state_kernel, g, smem)) return rc;
    wab_save_state_kernel<<<(unsigned)((n + kStateEnvs - 1) / kStateEnvs), kStateThreads, smem, (cudaStream_t)stream>>>(
        h->P, h->st, g, state_fingerprint(h), h->cfg.food_mode == WAB_FOOD_F64, d_slots, n, (uint4*)d_records);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab_vec_load_state(WabVec* h, const void* d_records, const int32_t* d_slots, int64_t n, WabObs obs,
                       int32_t* d_rejected, void* stream) {
    if (!h || !d_records || !d_rejected) return fail(WAB_E_NULL, "null argument");
    if (int rc = check_ptr_align(d_records, "d_records")) return rc;
    if (n < 0 || (!d_slots && n > h->n)) return fail(WAB_E_CONFIG, "without d_slots, n must be at most the number of envs");
    const bool emit = obs.d_grids || obs.d_food || obs.d_role || obs.d_status;
    if (emit) {
        if (!obs.d_food || !obs.d_role || !obs.d_status) return fail(WAB_E_NULL, "null argument");
        if (int rc = check_grids(h, obs.d_grids)) return rc;
    }
    DeviceGuard guard(h->device);
    h->started = true;
    cudaStream_t s = (cudaStream_t)stream;
    WAB_CUDA(cudaMemsetAsync(d_rejected, 0, sizeof(int32_t), s));
    if (n > 0) {
        const RecGeo g = rec_geo(h);
        const int f64 = h->cfg.food_mode == WAB_FOOD_F64;
        wab_validate_state_kernel<<<(unsigned)((n + kStateThreads - 1) / kStateThreads), kStateThreads, 0, s>>>(
            h->P, g, state_fingerprint(h), f64, h->n, (const uint32_t*)d_records, d_slots, n, d_rejected);
        WAB_CUDA(cudaGetLastError());
        size_t smem;
        if (int rc = state_smem((const void*)wab_load_state_kernel, g, smem)) return rc;
        wab_load_state_kernel<<<(unsigned)((n + kStateEnvs - 1) / kStateEnvs), kStateThreads, smem, s>>>(
            h->P, h->st, g, f64, (const uint4*)d_records, d_slots, n, d_rejected);
        WAB_CUDA(cudaGetLastError());
    }
    if (!emit) return WAB_OK;
    // observations from the reset kernels with nothing to reset: every env re-emits what its (loaded) state implies
    if (!h->d_zero_mask) {
        WAB_CUDA(cudaMalloc(&h->d_zero_mask, (size_t)h->n));
        WAB_CUDA(cudaMemsetAsync(h->d_zero_mask, 0, (size_t)h->n, s));
    }
    return wab_vec_reset(h, h->d_zero_mask, obs, stream);
}

int wab_vec_set_stats(WabVec* h, const int64_t* h_in8, void* stream) {
    if (!h || !h_in8) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    cudaStream_t s = (cudaStream_t)stream;
    WAB_CUDA(cudaMemsetAsync(h->st.wstats, 0, 64 * (size_t)h->stat_rows, s));
    WAB_CUDA(cudaMemcpyAsync(h->st.wstats, h_in8, 64, cudaMemcpyHostToDevice, s));
    return WAB_OK;
}

}  // extern "C"
