// wab2_kernels.cuh — Environment 2.0 world-turn kernels and their C ABI (included by wab_kernels.cu).
//
// One thread per world. The world's entities (three words each) are staged in shared memory with the thread
// index as the fastest dimension (bank-conflict free), every entity acts in turn exactly as the reference driver
// loop does (get_obs(i) then take_action(i, a), Env2Tests.py:46-88), and for each acting entity the 32 worlds
// of a warp publish their (2R+1)^2 x 3 one-hot windows together: every lane sets the bits of its own window in a
// shared-memory bit stream, then the warp expands the 32 streams with coalesced 16-byte streaming stores.
#pragma once

namespace {

struct State2Ptrs {
    uint32_t* ent;      // entity words (wab2_core.cuh): word f (0 object coords, 1 table row, 2 food) of entity k of world i
                        // at ent[k * stride_ent + f * stride_word + i * stride_world]
    uint32_t* episode;  // [N]
    uint32_t* turn;     // [N]
    int64_t n;
    int64_t stride_ent, stride_word, stride_world;   // [E][3][N] (thread per world: 3n, n, 1) or [N][3][E] (warp per world: 1, E, 3E)
};
struct Out2Ptrs {       // thread per world: entity-major (the 32 worlds of a warp are contiguous); warp per world: world-major
    uint8_t* planes;    // [A][N][3][S][S] | [N][A][3][S][S] u8, or null
    int32_t* internal;  // [A][N][5] | [N][A][5], or null
    float* reward;      // [A][N] | [N][A]
    uint8_t* done;      // [A][N] | [N][A]
};

// thread-per-world kernels: table rows and food are staged in shared memory, object coords are used in place
__device__ __forceinline__ void bind_world(const State2Ptrs& st, int64_t idx, World2& W) {
    W.obj = st.ent + idx * st.stride_world; W.ostride = st.stride_ent;
}
__device__ __forceinline__ void load_world(const Params2& P, const State2Ptrs& st, int64_t idx, World2& W) {
    bind_world(st, idx, W);
    for (int k = 0; k < P.n_entities; ++k) {
        W.base[(2 * k) * W.stride] = st.ent[k * st.stride_ent + st.stride_word + idx * st.stride_world];
        W.base[(2 * k + 1) * W.stride] = st.ent[k * st.stride_ent + 2 * st.stride_word + idx * st.stride_world];
    }
    W.episode = st.episode[idx]; W.turn = st.turn[idx];
    W.env_id = (uint32_t)(P.env_id_base + (uint64_t)idx);
}
__device__ __forceinline__ void store_world(const Params2& P, const State2Ptrs& st, int64_t idx, const World2& W) {
    for (int k = 0; k < P.n_entities; ++k) {
        st.ent[k * st.stride_ent + st.stride_word + idx * st.stride_world] = W.base[(2 * k) * W.stride];
        st.ent[k * st.stride_ent + 2 * st.stride_word + idx * st.stride_world] = W.base[(2 * k + 1) * W.stride];
    }
    st.episode[idx] = W.episode; st.turn[idx] = W.turn;
}

// mode 0: create entities; mode 1: reset_environment
__global__ void wab2_init_kernel(const __grid_constant__ Params2 P, const State2Ptrs st, const int mode) {
    extern __shared__ uint32_t smem2[];
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= st.n) return;
    World2 W;
    W.base = smem2 + threadIdx.x; W.stride = blockDim.x;
    if (mode == 0) {
        bind_world(st, idx, W);
        W.env_id = (uint32_t)(P.env_id_base + (uint64_t)idx);
        world2_create(P, W);
    } else {
        load_world(P, st, idx, W);
        world2_reset(P, W);
    }
    store_world(P, st, idx, W);
}

// One world turn: every entity observes (acting entities only, optional) and acts, in id order.
__global__ void wab2_turn_kernel(const __grid_constant__ Params2 P, const State2Ptrs st,
                                 const uint8_t* __restrict__ actions, const Out2Ptrs out, const int stream_words) {
    extern __shared__ uint32_t smem2[];
    const int bs = blockDim.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t idx = (int64_t)blockIdx.x * bs + threadIdx.x;
    const int64_t n = st.n;
    const bool active = idx < n;
    const int64_t warp_first = idx - lane;
    const int n_valid = (int)((n - warp_first) < 32 ? (n - warp_first > 0 ? n - warp_first : 0) : 32);
    uint32_t* ents = smem2;                                          // [2E][bs] table rows and food
    uint32_t* streams = ents + 2 * P.n_entities * bs;                // [warps][stream_words]: one stream per warp
    uint2* lut = reinterpret_cast<uint2*>(streams + (((bs >> 5) * stream_words + 1) & ~1));
    build_lut(lut);
    World2 W;
    W.base = ents + threadIdx.x; W.stride = bs;
    if (active) load_world(P, st, idx, W);
    const int S = 2 * P.window_r + 1, obs_bytes = 3 * S * S, A = P.n_acting;
    uint32_t* stream = streams + warp * stream_words;
    for (int a = 0; a < P.n_entities; ++a) {
        const bool acting = a < A;
        const int64_t o = (int64_t)a * n + idx;                       // [A][N] outputs
        if (acting && (out.planes || out.internal)) {
            const int64_t first_byte = ((int64_t)a * n + warp_first) * obs_bytes;   // the warp's 32 windows are contiguous
            const int off = out.planes ? obs_align_off(out.planes + first_byte) : 0;
            int32_t internal[5] = {0, 0, 0, 0, 0};
            if (out.planes) {
                for (int k = lane; k < stream_words; k += 32) stream[k] = 0u;
                __syncwarp();
            }
            if (active) {
                if (out.planes) {
                    world2_observe(P, W, a, stream, off + lane * obs_bytes, internal);
                } else {
                    const uint32_t obj = w2_obj(W, a), atab = w2_tab(W, a);
                    const uint32_t at = entity_type(P, a);
                    internal[0] = unpack_x(obj); internal[1] = unpack_y(obj); internal[2] = (int32_t)w2_food(W, a);
                    internal[3] = at == T_BUSH ? 0 : (int32_t)((atab >> 17) & 1u);
                    internal[4] = at == T_BUSH ? 0 : (int32_t)((atab >> 18) & 3u);
                }
                if (out.internal) {
                    int32_t* dst = out.internal + o * 5;
                    dst[0] = internal[0]; dst[1] = internal[1]; dst[2] = internal[2]; dst[3] = internal[3]; dst[4] = internal[4];
                }
            }
            if (out.planes) {
                __syncwarp();
                stream_flush(stream, lut, out.planes + (first_byte - off), off, off + obs_bytes * n_valid, lane);
                __syncwarp();
            }
        }
        if (active) {
            float reward; uint32_t done;
            world2_act(P, W, a, acting ? (uint32_t)actions[o] : 0u, reward, done);
            if (acting) {
                out.reward[o] = reward;
                out.done[o] = (uint8_t)done;
            }
        }
    }
    if (active) store_world(P, st, idx, W);
}

}  // namespace

#include "wab2_grid.cuh"

typedef void (*GridKernel)(const Params2, const State2Ptrs, const uint8_t*, const Out2Ptrs);
static GridKernel grid_kernel_for(const Params2& P) {
    const bool h64 = P.height == 64, narrow = 2 * P.window_r + 1 < 15;
    return h64 ? (narrow ? wab2_grid_turn_kernel<true, true> : wab2_grid_turn_kernel<true, false>)
               : (narrow ? wab2_grid_turn_kernel<false, true> : wab2_grid_turn_kernel<false, false>);
}

struct Wab2World {
    Wab2Config cfg;
    Params2 P;
    State2Ptrs st;
    int device;
    int64_t n;
    void* slab;
    int bs, stream_words;
    size_t smem_turn, smem_init;
    bool grid;            // warp-per-world kernel with occupancy planes (wab2_grid.cuh)
};

extern "C" {

int wab2_create(const Wab2Config* cfg, int64_t n_envs, uint64_t seed, uint64_t env_id_base, int32_t device, Wab2World** out) {
    if (!cfg || !out) return fail(WAB_E_NULL, "null argument");
    *out = nullptr;
    if (cfg->abi_version != WAB_ABI_VERSION) return fail(WAB_E_CONFIG, "Wab2Config.abi_version mismatch");
    const int E = cfg->n_ostriches + cfg->n_wolves + cfg->n_bushes;
    if (cfg->width < 1 || cfg->height < 1 || cfg->width > 254 || cfg->height > 254) return fail(WAB_E_CONFIG, "world size must be in [1, 254]");
    if (cfg->n_ostriches < 0 || cfg->n_wolves < 0 || cfg->n_bushes < 0 || E < 1 || E > 1024) return fail(WAB_E_CONFIG, "entity counts out of range");
    if (cfg->n_ostriches + cfg->n_wolves < 1) return fail(WAB_E_CONFIG, "at least one acting entity is required");
    if (cfg->window_radius < 0 || cfg->window_radius > 15) return fail(WAB_E_CONFIG, "window_radius must be in [0, 15]");
    if (cfg->lookout_view_radius < 0 || cfg->gatherer_view_radius < 0 || cfg->wolf_view_radius < 0) return fail(WAB_E_CONFIG, "negative view radius");
    if (cfg->starting_role != 0 && cfg->starting_role != 1) return fail(WAB_E_UNSUPPORTED, "starting_role must be 0 or 1");
    if (n_envs < 1) return fail(WAB_E_CONFIG, "n_envs must be >= 1");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(WAB_E_NO_DEVICE, "no CUDA device: wab_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(WAB_E_CONFIG, "bad device ordinal");
    DeviceGuard guard(device);
    Wab2World* h = new (std::nothrow) Wab2World();
    if (!h) return fail(WAB_E_CUDA, "out of host memory");
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg; h->device = device; h->n = n_envs;
    Params2& P = h->P;
    fill_round_keys2(P, (uint32_t)seed, (uint32_t)(seed >> 32));
    P.width = cfg->width; P.height = cfg->height; P.n_ostriches = cfg->n_ostriches; P.n_wolves = cfg->n_wolves;
    P.n_bushes = cfg->n_bushes; P.n_entities = E; P.n_acting = cfg->n_ostriches + cfg->n_wolves;
    P.lookout_r = cfg->lookout_view_radius; P.gatherer_r = cfg->gatherer_view_radius; P.wolf_r = cfg->wolf_view_radius;
    P.window_r = cfg->window_radius; P.starting_role = cfg->starting_role; P.ostrich_food = cfg->ostrich_starting_food;
    P.wolf_food = cfg->wolf_starting_food; P.wolf_eat_gain = cfg->wolf_food_for_eating_ostrich;
    P.bush_food = cfg->food_per_bush; P.bush_given = cfg->food_given_per_turn; P.env_id_base = env_id_base;
    const int S = 2 * cfg->window_radius + 1;
    const int rads[3] = {cfg->lookout_view_radius, cfg->gatherer_view_radius, cfg->wolf_view_radius};
    for (int s3 = 0; s3 < 3; ++s3)
        for (int d = 0; d < 16; ++d) {
            int m = 0;
            while (d <= rads[s3] && (m + 1) * (m + 1) + d * d <= rads[s3] * rads[s3]) ++m;
            P.halfwidth[s3][d] = (uint8_t)m;
        }
    const int rmax = rads[0] > rads[1] ? (rads[0] > rads[2] ? rads[0] : rads[2]) : (rads[1] > rads[2] ? rads[1] : rads[2]);
    // every window fits the world once -> occupancy-plane kernel, one warp per world
    h->grid = cfg->window_radius >= rmax && cfg->width >= S && cfg->height >= S && cfg->width <= 64 && cfg->height <= 64 &&
              (E > 96 || getenv("WAB2_GRID") != nullptr) && getenv("WAB2_NO_GRID") == nullptr;   // small worlds: thread per world is faster
    h->stream_words = h->grid ? (3 * S * S + 15 + 31) / 32 + 1 : (32 * 3 * S * S + 31 + 31) / 32 + 1;   // thread per world: 32-byte store grid
    // threads per block: as many as shared memory allows (3E state words + one bit stream per thread)
    int max_smem = 48 * 1024;
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    // 64-thread CTAs: a 65,536-world batch is 1,024 CTAs = 6.9 per SM (12 or 14 warps), where 128-thread CTAs gave 3 or 4
    // per SM (12 or 16 warps) and the fuller SMs set the launch time: 3.19e8 -> 3.35e8 world turns/s (profiles/r2v_v2_bs.txt)
    int bs = 64;
    auto need = [&](int b) { return sizeof(uint32_t) * ((size_t)2 * E * b + (size_t)(((b >> 5) * h->stream_words + 1) & ~1) + 512); };
    if (const char* eb = getenv("WAB2_BS")) { const int v = atoi(eb); if (v == 32 || v == 64 || v == 128) bs = v; }   // A/B runs
    while (bs > 32 && need(bs) > (size_t)max_smem / 2) bs >>= 1;
    if (need(bs) > (size_t)max_smem) { delete h; return fail(WAB_E_UNSUPPORTED, "too many entities for the shared-memory staging"); }
    h->bs = bs; h->smem_turn = need(bs); h->smem_init = sizeof(uint32_t) * (size_t)2 * E * bs;
    cudaError_t e = cudaSuccess;
    if (h->grid) {
        h->smem_turn = sizeof(uint32_t) * ((size_t)4 * grid_geom(E, P.n_acting, cfg->width, S).total + 512);
        e = cudaFuncSetAttribute(grid_kernel_for(h->P), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_turn);
    } else
        e = cudaFuncSetAttribute(wab2_turn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_turn);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(wab2_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_init);
    const size_t n = (size_t)n_envs;
    size_t o = 0;
    const size_t o_ent = o; o = align_up(o + 4 * n * 3 * (size_t)E, 256);
    const size_t o_ep = o; o = align_up(o + 4 * n, 256);
    const size_t o_turn = o; o = align_up(o + 4 * n, 256);
    if (e == cudaSuccess) e = cudaMalloc(&h->slab, o);
    if (e == cudaSuccess) e = cudaMemset(h->slab, 0, o);
    if (e != cudaSuccess) { if (h->slab) cudaFree(h->slab); delete h; return cuda_fail(e, "wab2_create"); }
    uint8_t* base = (uint8_t*)h->slab;
    h->st.ent = (uint32_t*)(base + o_ent); h->st.episode = (uint32_t*)(base + o_ep); h->st.turn = (uint32_t*)(base + o_turn);
    h->st.n = n_envs;
    h->st.stride_ent = h->grid ? 1 : 3 * n_envs;
    h->st.stride_word = h->grid ? E : n_envs;
    h->st.stride_world = h->grid ? 3 * E : 1;
    wab2_init_kernel<<<(unsigned)((n_envs + bs - 1) / bs), bs, h->smem_init, 0>>>(h->P, h->st, 0);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { cudaFree(h->slab); delete h; return cuda_fail(e, "wab2_init_kernel"); }
    *out = h;
    return WAB_OK;
}

void wab2_destroy(Wab2World* h) {
    if (!h) return;
    DeviceGuard guard(h->device);
    if (h->slab) cudaFree(h->slab);
    delete h;
}

int wab2_kernel_kind(const Wab2World* h) { return h && h->grid ? 1 : 0; }
int wab2_output_layout(const Wab2World* h) { return h && h->grid ? 1 : 0; }

int wab2_reset(Wab2World* h, void* stream) {
    if (!h) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    wab2_init_kernel<<<(unsigned)((h->n + h->bs - 1) / h->bs), h->bs, h->smem_init, (cudaStream_t)stream>>>(h->P, h->st, 1);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab2_turn(Wab2World* h, const uint8_t* d_actions, uint8_t* d_planes, int32_t* d_internal, float* d_reward,
              uint8_t* d_done, void* stream) {
    if (!h || !d_actions || !d_reward || !d_done) return fail(WAB_E_NULL, "null argument");
    if (d_planes) if (int rc = check_ptr_align(d_planes, "d_planes")) return rc;
    DeviceGuard guard(h->device);
    Out2Ptrs out{d_planes, d_internal, d_reward, d_done};
    if (h->grid)
        grid_kernel_for(h->P)<<<(unsigned)((h->n + 3) / 4), 128, h->smem_turn, (cudaStream_t)stream>>>(h->P, h->st, d_actions, out);
    else
        wab2_turn_kernel<<<(unsigned)((h->n + h->bs - 1) / h->bs), h->bs, h->smem_turn, (cudaStream_t)stream>>>(
            h->P, h->st, d_actions, out, h->stream_words);
    WAB_CUDA(cudaGetLastError());
    return WAB_OK;
}

int wab2_export_state(Wab2World* h, int32_t* out9, int32_t* turn, int32_t* episode, void* stream) {
    if (!h || !out9) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    WAB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    const size_t n = (size_t)h->n;
    const int E = h->P.n_entities;
    uint32_t* ent = new uint32_t[n * 3 * E];
    uint32_t* tr = new uint32_t[n];
    cudaError_t e = cudaMemcpy(ent, h->st.ent, 4 * n * 3 * E, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(tr, h->st.turn, 4 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && episode) e = cudaMemcpy(episode, h->st.episode, 4 * n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess)
        for (size_t i = 0; i < n; ++i) {
            if (turn) turn[i] = (int32_t)tr[i];
            for (int k = 0; k < E; ++k) {
                const size_t se = (size_t)h->st.stride_ent, sw = (size_t)h->st.stride_word, si = (size_t)h->st.stride_world;
                const uint32_t obj = ent[k * se + i * si], tab = ent[k * se + sw + i * si], food = ent[k * se + 2 * sw + i * si];
                int32_t* o = out9 + (i * E + k) * 9;
                o[0] = (int32_t)entity_type(h->P, k); o[1] = unpack_x(obj); o[2] = unpack_y(obj);
                o[3] = (int32_t)(tab & 0xFFu); o[4] = (int32_t)((tab >> 8) & 0xFFu); o[5] = (int32_t)((tab >> 16) & 1u);
                o[6] = (int32_t)food; o[7] = (int32_t)((tab >> 17) & 1u); o[8] = (int32_t)((tab >> 18) & 3u);
            }
        }
    delete[] ent; delete[] tr;
    if (e != cudaSuccess) return cuda_fail(e, "wab2_export_state");
    return WAB_OK;
}

int wab2_import_state(Wab2World* h, const int32_t* in9, const int32_t* turn, const int32_t* episode, void* stream) {
    if (!h || !in9) return fail(WAB_E_NULL, "null argument");
    DeviceGuard guard(h->device);
    WAB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    const size_t n = (size_t)h->n;
    const int E = h->P.n_entities;
    const size_t se = (size_t)h->st.stride_ent, sw = (size_t)h->st.stride_word, si = (size_t)h->st.stride_world;
    uint32_t* ent = new uint32_t[n * 3 * E];
    int bad = 0;
    for (size_t i = 0; i < n && !bad; ++i)
        for (int k = 0; k < E; ++k) {
            const int32_t* o = in9 + (i * E + k) * 9;
            if (o[0] != (int32_t)entity_type(h->P, k) || o[3] < 0 || o[3] > 255 || o[4] < 0 || o[4] > 255 || o[6] < 0 ||
                o[1] < -32768 || o[1] > 32767 || o[2] < -32768 || o[2] > 32767) { bad = 1; break; }
            ent[k * se + i * si] = pack_xy(o[1], o[2]);
            ent[k * se + sw + i * si] = tab_pack((uint32_t)o[3], (uint32_t)o[4], o[5] ? 1u : 0u, (uint32_t)o[7] & 1u, (uint32_t)o[8] & 3u);
            ent[k * se + 2 * sw + i * si] = (uint32_t)o[6];
        }
    cudaError_t e = cudaSuccess;
    if (!bad) e = cudaMemcpy(h->st.ent, ent, 4 * n * 3 * E, cudaMemcpyHostToDevice);
    if (!bad && e == cudaSuccess && turn) e = cudaMemcpy(h->st.turn, turn, 4 * n, cudaMemcpyHostToDevice);
    if (!bad && e == cudaSuccess && episode) e = cudaMemcpy(h->st.episode, episode, 4 * n, cudaMemcpyHostToDevice);
    delete[] ent;
    if (bad) return fail(WAB_E_CONFIG, "wab2_import_state: entity type order or value range does not fit the handle");
    if (e != cudaSuccess) return cuda_fail(e, "wab2_import_state");
    return WAB_OK;
}

}  // extern "C"
