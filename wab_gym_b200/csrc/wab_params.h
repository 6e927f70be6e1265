// wab_params.h — host-side validation of WabConfig and construction of the kernel Params.
// Shared by the C ABI (wab_kernels.cu) and the host-compiled logic test (tests/hostsim).
#pragma once
#include <string.h>

#include <string>

#include "../../include/wab_b200.h"
#include "wab_core.cuh"

namespace wab {

inline void fill_round_keys(Params& P, uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) { P.rk0[r] = k0; P.rk1[r] = k1; k0 += PHILOX_W0; k1 += PHILOX_W1; }
}

// Fingerprint of what a saved env state depends on (wab_vec_state_fingerprint): every WabConfig field by VALUE (the
// struct's padding bytes are undefined), the bush threshold table, the seed and the kernel kind. env_id_base and n_envs
// are left out, so records move between shard layouts.
inline uint64_t fp_mix(uint64_t h, uint64_t v) {
    h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
    h ^= h >> 30; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 27; h *= 0x94D049BB133111EBull; h ^= h >> 31;
    return h;
}
inline uint64_t fp_f64(double d) { uint64_t v; memcpy(&v, &d, 8); return v; }
inline uint64_t config_fingerprint(const WabConfig& c, const uint32_t* bush_thr, int32_t n_bush_thr, uint64_t seed, bool generic) {
    uint64_t h = 0x5741425354415445ull;
    const int64_t ints[] = {c.abi_version, c.width, c.height, c.max_turns, c.wolf_spawn_margin, c.n_actions,
                            c.lookout_only, c.restrict_view, c.wolves, c.wolves_can_move, c.god_mode, c.starting_role,
                            c.food_mode, c.auto_reset, c.food_int_start, c.food_int_inc, c.food_int_max, c.wolf_cap, c.log_cap};
    for (int64_t v : ints) h = fp_mix(h, (uint64_t)v);
    for (int a = 0; a < WAB_MAX_ACTIONS; ++a)
        h = fp_mix(h, (uint64_t)(uint8_t)c.action_dx[a] | (uint64_t)(uint8_t)c.action_dy[a] << 8 | (uint64_t)(uint8_t)c.action_role[a] << 16);
    h = fp_mix(h, fp_f64(c.food_start)); h = fp_mix(h, fp_f64(c.food_inc));
    h = fp_mix(h, fp_f64(c.food_dec)); h = fp_mix(h, fp_f64(c.food_obs_scale));
    for (int k = 0; k < 32; ++k) { h = fp_mix(h, c.spawn_cdf[k]); h = fp_mix(h, c.init_cdf[k]); }
    h = fp_mix(h, c.thr_keep);
    for (int k = 0; k < 8; ++k) { uint32_t v; memcpy(&v, &c.reward_table[k], 4); h = fp_mix(h, v); }
    for (int k = 0; k < 4; ++k) h = fp_mix(h, (uint64_t)c.mask_lookout[k] | (uint64_t)c.mask_gatherer[k] << 32);
    h = fp_mix(h, (uint64_t)n_bush_thr);
    for (int32_t k = 0; k < n_bush_thr; ++k) h = fp_mix(h, bush_thr[k]);
    h = fp_mix(h, seed);
    return fp_mix(h, generic ? 1u : 0u);
}

inline int validate_config(const WabConfig* cfg, int32_t n_bush_thr, int64_t n_envs, std::string& err) {
    auto fail = [&err](int code, const char* msg) { err = msg; return code; };
    if (cfg->abi_version != WAB_ABI_VERSION) return fail(WAB_E_CONFIG, "WabConfig.abi_version mismatch");
    if (cfg->width % 2 == 0 || cfg->height % 2 == 0)
        return fail(WAB_E_CONFIG, "width and height must be odd numbers");       // wab_env.py:147-148
    if (cfg->width < 1 || cfg->height < 1 || cfg->width > 31 || cfg->height > 31)
        return fail(WAB_E_UNSUPPORTED, "viewports up to 31 x 31 are implemented");
    if (cfg->wolf_spawn_margin < 1 || cfg->wolf_spawn_margin > 2)
        return fail(WAB_E_UNSUPPORTED, "wolf_spawn_margin 1 and 2 are implemented");
    if (cfg->restrict_view && (cfg->width != VIEW || cfg->height != VIEW))
        return fail(WAB_E_UNSUPPORTED, "restrict_view exists for the 11 x 11 viewport only (the reference's tile masks are 11 x 11 literals)");
    if (n_envs < 1) return fail(WAB_E_CONFIG, "n_envs must be >= 1");
    for (int k = 1; k < 32; ++k)
        if (cfg->spawn_cdf[k] < cfg->spawn_cdf[k - 1] || cfg->init_cdf[k] < cfg->init_cdf[k - 1])
            return fail(WAB_E_CONFIG, "binomial-first tables must be non-decreasing");
    if (cfg->n_actions < 1 || cfg->n_actions > WAB_MAX_ACTIONS) return fail(WAB_E_CONFIG, "n_actions out of range");
    if (cfg->max_turns < 1 || cfg->max_turns > 30000) return fail(WAB_E_CONFIG, "max_turns must be in [1, 30000]");
    if (cfg->wolf_cap < 1 || cfg->wolf_cap > 64) return fail(WAB_E_CONFIG, "wolf_cap must be in [1, 64]");
    if (cfg->log_cap < 1 || cfg->log_cap > 255) return fail(WAB_E_CONFIG, "log_cap must be in [1, 255]");
    if (n_bush_thr < 0 || n_bush_thr > 255) return fail(WAB_E_UNSUPPORTED, "max_berries_per_bush above 255");
    if (cfg->food_mode != WAB_FOOD_F64 && cfg->food_mode != WAB_FOOD_INT) return fail(WAB_E_CONFIG, "food_mode");
    if (cfg->food_mode == WAB_FOOD_INT &&
        (cfg->food_int_max < 1 || cfg->food_int_max > 255 || cfg->food_int_start < 0 ||
         cfg->food_int_start > cfg->food_int_max || cfg->food_int_inc < 0 || !cfg->auto_reset || cfg->food_start < 0))
        return fail(WAB_E_CONFIG, "integer food mode needs a host proof, fixed starting_food and auto_reset");
    if (cfg->food_obs_scale <= 0 || cfg->food_obs_scale > 255) return fail(WAB_E_CONFIG, "turns_to_empty_food must be in (0, 255]");
    for (int a = 0; a < cfg->n_actions; ++a) {
        if (cfg->action_dx[a] < -1 || cfg->action_dx[a] > 1 || cfg->action_dy[a] < -1 || cfg->action_dy[a] > 1 ||
            (cfg->action_dx[a] != 0 && cfg->action_dy[a] != 0) || cfg->action_role[a] < -1 || cfg->action_role[a] > 1)
            return fail(WAB_E_CONFIG, "action table rows must be unit axis moves with role in {-1, 0, 1}");
    }
    return WAB_OK;
}

// bush_thr must already be the pointer the kernels will dereference (device pointer for the GPU).
inline void params_from_config(const WabConfig& c, const uint32_t* bush_thr_host, int32_t n_bush_thr, uint64_t seed,
                               uint64_t env_id_base, Params& P) {
    const WabConfig* cfg = &c;
    const uint32_t* bush_thr = bush_thr_host;
    memset(&P, 0, sizeof(P));
    fill_round_keys(P, (uint32_t)seed, (uint32_t)(seed >> 32));
    {
        uint32_t k2 = (uint32_t)(seed ^ (seed >> 32));
        for (int r = 0; r < 10; ++r) { P.rk2[r] = k2; k2 += PHILOX_W0; }
    }
    P.n_bush_thr = (uint32_t)n_bush_thr;
    P.thr_bush1 = n_bush_thr > 0 ? bush_thr[0] : 0xFFFFFFFFu;
    P.thr_bush2 = n_bush_thr > 1 ? bush_thr[1] : 0xFFFFFFFFu;
    for (int k = 0; k < 32; ++k) { P.spawn_cdf[k] = cfg->spawn_cdf[k]; P.init_cdf[k] = cfg->init_cdf[k]; }
    P.thr_keep = cfg->thr_keep;
    P.act_tbl = 0;
    for (int a = 0; a < cfg->n_actions; ++a) {
        const uint64_t code = (uint64_t)(cfg->action_dx[a] + 1) | ((uint64_t)(cfg->action_dy[a] + 1) << 2) |
                              ((uint64_t)(cfg->action_role[a] + 1) << 4);
        P.act_tbl |= code << (8 * a);
    }
    P.n_actions = cfg->n_actions; P.max_turns = cfg->max_turns;
    P.food_int_start = cfg->food_int_start; P.food_int_inc = cfg->food_int_inc; P.food_int_max = cfg->food_int_max;
    P.wolf_cap = cfg->wolf_cap; P.log_cap = cfg->log_cap;
    P.lookout_only = cfg->lookout_only; P.restrict_view = cfg->restrict_view; P.wolves = cfg->wolves;
    P.wolves_can_move = cfg->wolves_can_move; P.god_mode = cfg->god_mode; P.auto_reset = cfg->auto_reset;
    P.starting_role = cfg->starting_role;
    P.food_random = cfg->food_start < 0 ? 1 : 0;
    P.food_start = cfg->food_start; P.food_inc = cfg->food_inc; P.food_dec = cfg->food_dec;
    P.food_obs_scale = cfg->food_obs_scale;
    for (int k = 0; k < 8; ++k) P.reward_table[k] = cfg->reward_table[k];
    for (int k = 0; k < 4; ++k) { P.mask_look[k] = cfg->mask_lookout[k]; P.mask_gath[k] = cfg->mask_gatherer[k]; }
    P.env_id_base = env_id_base;

}

}  // namespace wab
