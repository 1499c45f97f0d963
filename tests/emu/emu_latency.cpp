// TEST-ONLY warp emulation of an env step with per-robot command latency (plen_set_env_latency).  Builds on the harness of
// emu_warp.cpp (the product's device source compiled for the host, 32 threads + barriers standing in for one warp) and adds
// emu_latency_source (the device selection function itself), emu_step_latency (the k_dyn prologue with a history ring, the
// ticks and env_post, the way plen_b200.cu runs a step once the ring exists) and emu_post (env_post alone, so that a reference
// can drive emu_tick tick by tick and finish the step the same way).  Never linked into the product library.
#include <algorithm>

#include "emu_warp.cpp"

namespace {
// as run_ticks of emu_warp.cpp for the substeps of one env step: tick 0 derives the raw targets from the actions (tgt, [n][18])
// and records them in the robot's ring row; every tick applies the targets latency_source selects, as k_dyn does
void run_step_latency(const DevConfig &dc, const EnvRanges &er, const float *tab, float *records, const float *actions,
                      float *tgt, float *ring, const int *ticks, int n, int lane) {
    static WarpScratch ws;
    static std::vector<float> srec, srx, Gs(PLEN_SOLVE_ROBOTS * PLEN_GS_WORDS);
    static std::vector<uint8_t> keys;
    if (lane == 0) { srec.assign((size_t)n * SR_WORDS, 0.0f); srx.assign((size_t)n * XR_WORDS, 0.0f); keys.assign(n, 0); }
    bar();
    const int max_ticks = PLEN_MAX_LATENCY_STEPS * dc.substeps;
    for (int t = 0; t < dc.substeps; t++) {
        for (int e = 0; e < n; e++) {
            LaneState L;
            load_record(records + 96 * e, ws, L, lane);
            const int ept = std::max((int)records[96 * e + W_EPT], 0);
            const int d = std::min(std::max(ticks[e], 0), max_ticks);          // the setter's clamp
            const int src = latency_source(d, t, dc.substeps, ept);
            float *row = ring + (size_t)e * LAT_WORDS;
            if (lane >= 6 && lane < 24) {
                const int j = lane - 6;
                if (t == 0) {
                    tgt[18 * e + j] = agent_target(dc, er, j, actions[18 * e + j]);
                    row[32 * latency_slot(ept, 0) + lane] = tgt[18 * e + j];
                }
                L.tgt = src == 0 ? tgt[18 * e + j] : src < 0 ? 0.0f : row[32 * latency_slot(ept, src) + lane];
            }
            tick_dynamics(dc, tab, ws, L, lane, srec.data() + (size_t)e * SR_WORDS, keys.data() + e, nullptr,
                          srx.data() + (size_t)e * XR_WORDS, nullptr);
        }
        for (int b = 0; b < n; b += PLEN_SOLVE_ROBOTS) {
            const int r = b + (lane >> 2);
            const bool valid = r < n;
            const int rr = valid ? r : 0;
            bool anyx = false;
            for (int k = b; k < b + PLEN_SOLVE_ROBOTS && k < n; k++) anyx = anyx || keys[k] >= PLEN_KEY_EXT;
            if (anyx) {
                const int nx = (valid && keys[rr] >= PLEN_KEY_EXT) ? (int)srx[(size_t)rr * XR_WORDS + XR_NX] : 0;
                solve_tick<1>(dc, srec.data() + (size_t)rr * SR_WORDS, Gs.data() + (lane >> 2) * PLEN_GS_WORDS, records + 96 * rr, lane, valid,
                              srx.data() + (size_t)rr * XR_WORDS, nx);
            } else {
                solve_tick<0>(dc, srec.data() + (size_t)rr * SR_WORDS, Gs.data() + (lane >> 2) * PLEN_GS_WORDS, records + 96 * rr, lane, valid);
            }
            bar();
        }
    }
}

void post(const DevConfig &dc, const float *tab, float *records, int n, float *obs, float *reward, uint8_t *done,
          uint8_t *timeout, float *terminal_obs, const float *snapshot, int lane) {
    static WarpScratch ws;
    for (int e = 0; e < n; e++) {
        LaneState L;
        load_record(records + 96 * e, ws, L, lane);
        StepIO io{nullptr, obs + 26 * e, reward + e, done + e, timeout ? timeout + e : nullptr,
                  terminal_obs ? terminal_obs + 26 * e : nullptr, snapshot, nullptr};
        env_post(dc, tab, ws, L, lane, io);
        store_record(records + 96 * e, ws, L, lane);
    }
}

void setup(const plen_model *m, const plen_config *c, std::vector<float> &tab, std::vector<float> &hull, DevConfig &dc,
           EnvRanges &er) {
    tab.assign(T_ROWS * 32, 0.0f);
    build_table(m, c, tab.data());
    build_devconfig(m, c, &dc, &er);
    hull.resize(2 * PLEN_MAX_HULL * 3);
    for (size_t i = 0; i < hull.size(); i++) hull[i] = (&m->foot_hull[0][0][0])[i];
    dc.hull = hull.data();
}
}  // namespace

extern "C" {
int emu_latency_source(int d, int k, int S, int ep_t) { return latency_source(d, k, S, ep_t); }
int emu_latency_slot(int ep_t, int s) { return latency_slot(ep_t, s); }

// one env step of n robots with command latency: records [n][96], actions [n][18] (agent space), tgt [n][18] (out: the raw
// targets of this step), ring [n][LAT_WORDS] (in / out), ticks [n]; outputs as emu_step
void emu_step_latency(const plen_model *m, const plen_config *c, float *records, const float *actions, float *tgt, float *ring,
                      const int *ticks, int n, float *obs, float *reward, uint8_t *done, uint8_t *timeout, float *terminal_obs,
                      const float *snapshot) {
    std::vector<float> tab, hull;
    DevConfig dc; EnvRanges er;
    setup(m, c, tab, hull, dc, er);
    run_warp([&](int lane) {
        run_step_latency(dc, er, tab.data(), records, actions, tgt, ring, ticks, n, lane);
        post(dc, tab.data(), records, n, obs, reward, done, timeout, terminal_obs, snapshot, lane);
    });
}

// env_post alone (what k_post runs after the last tick of a step)
void emu_post(const plen_model *m, const plen_config *c, float *records, int n, float *obs, float *reward, uint8_t *done,
              uint8_t *timeout, float *terminal_obs, const float *snapshot) {
    std::vector<float> tab, hull;
    DevConfig dc; EnvRanges er;
    setup(m, c, tab, hull, dc, er);
    run_warp([&](int lane) { post(dc, tab.data(), records, n, obs, reward, done, timeout, terminal_obs, snapshot, lane); });
}
}
