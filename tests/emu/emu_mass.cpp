// TEST-ONLY warp emulation of the MASS instance of tick_dynamics (k_dyn<true>: per-robot mass rows, plen_set_env_mass).
// Builds on the harness of emu_warp.cpp (the product's device source compiled for the host, 32 threads + barriers standing in
// for one warp) and adds one entry point, emu_tick_mass, which runs (k_dyn<true>, k_solve) x n_ticks the way plen_b200.cu
// launches them when mass rows are set.  Never linked into the product library.
#include "emu_warp.cpp"

namespace {
// as run_ticks of emu_warp.cpp, with the robot's mass row word in L.mass_w and the MASS instance of the dynamics
void run_ticks_mass(const DevConfig &dc, const float *tab, float *records, const float *tgt, const float *rows, int n,
                    int n_ticks, const DebugOut *dbg0, int lane) {
    static WarpScratch ws;
    static std::vector<float> srec, srx, Gs(PLEN_SOLVE_ROBOTS * PLEN_GS_WORDS);
    static std::vector<uint8_t> keys;
    if (lane == 0) { srec.assign((size_t)n * SR_WORDS, 0.0f); srx.assign((size_t)n * XR_WORDS, 0.0f); keys.assign(n, 0); }
    bar();
    for (int t = 0; t < n_ticks; t++) {
        for (int e = 0; e < n; e++) {
            LaneState L;
            load_record(records + 96 * e, ws, L, lane);
            if (lane >= 6 && lane < 24) L.tgt = tgt ? tgt[18 * e + lane - 6] : 0.0f;
            L.mass_w = rows[(size_t)e * MR_WORDS + lane];
            tick_dynamics<true>(dc, tab, ws, L, lane, srec.data() + (size_t)e * SR_WORDS, keys.data() + e,
                                (e == 0 && t == n_ticks - 1) ? dbg0 : nullptr, srx.data() + (size_t)e * XR_WORDS, nullptr);
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
}  // namespace

extern "C" {
// emu_tick with mass rows [n][MR_WORDS] (layout of plen_set_env_mass: word 0 and words 6..23 the body scales, 24..27 the payload)
void emu_tick_mass(const plen_model *m, const plen_config *c, float *records, const float *targets, const float *rows, int n,
                   int n_ticks, float *dbg_minv, float *dbg_pos, float *dbg_rot) {
    std::vector<float> tab(T_ROWS * 32);
    DevConfig dc; EnvRanges er;
    build_table(m, c, tab.data());
    build_devconfig(m, c, &dc, &er);
    std::vector<float> hull(2 * PLEN_MAX_HULL * 3);
    for (size_t i = 0; i < hull.size(); i++) hull[i] = (&m->foot_hull[0][0][0])[i];
    dc.hull = hull.data();
    DebugOut dbg{dbg_minv, dbg_pos, dbg_rot};
    run_warp([&](int lane) { run_ticks_mass(dc, tab.data(), records, targets, rows, n, n_ticks, dbg_minv ? &dbg : nullptr, lane); });
}
}
