// TEST-ONLY warp emulation of the per-robot observation noise (plen_set_env_obs_noise).  Builds on the harness of emu_warp.cpp
// (the product's device source compiled for the host) and exports the noise generator of plen_env.cuh and env_post's noise
// instance, as k_post runs it.  Never linked into the product library.
#include "emu_warp.cpp"

extern "C" {
// generator pieces for keys k[n]: hash32(k), the two float32 uniforms, the Gaussian, and the flip decision at probability p[i]
void emu_noise_draws(const uint64_t *k, const float32_t_ *p, int n, uint32_t *hash, float32_t_ *u1, float32_t_ *u2, double *normal,
                     uint8_t *flip) {
    for (int i = 0; i < n; i++) {
        hash[i] = noise_hash32(k[i]);
        u1[i] = (float32_t_)noise_u1(k[i]);
        u2[i] = (float32_t_)noise_u2(k[i]);
        normal[i] = (double)noise_normal(k[i]);
        flip[i] = noise_flip(k[i], p[i]) ? 1 : 0;
    }
}

uint64_t emu_noise_key(unsigned long long seed, long long gid, unsigned ctr, int stream, int word) {
    return obs_noise_key(obs_noise_base(seed, gid), ctr, stream, word);
}

// emu_step with the noise instance of env_post: rows [n][ON_WORDS] (updated: biases, counters), clean_obs / clean_tobs [n][26]
void emu_step_noise(const plen_model *m, const plen_config *c, float *records, const float *actions, int n, float *obs,
                    float *reward, uint8_t *done, uint8_t *timeout, float *terminal_obs, const float *snapshot, float *rows,
                    float *clean_obs, float *clean_tobs, unsigned long long seed, long long gid0) {
    std::vector<float> tab(T_ROWS * 32), tgt((size_t)n * 18);
    DevConfig dc; EnvRanges er;
    build_table(m, c, tab.data());
    build_devconfig(m, c, &dc, &er);
    std::vector<float> hull(2 * PLEN_MAX_HULL * 3);
    for (size_t i = 0; i < hull.size(); i++) hull[i] = (&m->foot_hull[0][0][0])[i];
    dc.hull = hull.data();
    for (int e = 0; e < n; e++)
        for (int j = 0; j < 18; j++) tgt[18 * e + j] = agent_target(dc, er, j, actions[18 * e + j]);
    static WarpScratch ws;
    run_warp([&](int lane) {
        run_ticks(dc, tab.data(), records, tgt.data(), n, dc.substeps, nullptr, lane);
        for (int e = 0; e < n; e++) {
            LaneState L;
            load_record(records + 96 * e, ws, L, lane);
            StepIO io{nullptr, obs + 26 * e, reward + e, done + e, timeout ? timeout + e : nullptr,
                      terminal_obs ? terminal_obs + 26 * e : nullptr, snapshot, nullptr, nullptr,
                      rows + (size_t)ON_WORDS * e, clean_obs + 26 * e, clean_tobs + 26 * e, obs_noise_base(seed, gid0 + e)};
            env_post<true>(dc, tab.data(), ws, L, lane, io);
            store_record(records + 96 * e, ws, L, lane);
        }
    });
}
}
