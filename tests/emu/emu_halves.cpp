// TEST-ONLY warp emulation of the two halves of a physics tick on their own: emu_dyn runs k_dyn's tick_dynamics over a batch
// and returns the solve records, extension records and sort keys; emu_solve runs k_solve's solve_tick on given records.
// Builds on the harness of emu_warp.cpp (the product's device source compiled for the host, 32 threads + barriers standing
// in for one warp), which stays as it is.  emu_dyn followed by emu_solve is emu_tick.  With -DPLEN_EMU_DOUBLE both run in
// float64, the reference the GPU's halves are checked against.  Never linked into the product library.
#include "emu_warp.cpp"

namespace {
struct HostTables {
    std::vector<float> tab, hull;
    DevConfig dc;
    EnvRanges er;
    HostTables(const plen_model *m, const plen_config *c) : tab(T_ROWS * 32), hull(2 * PLEN_MAX_HULL * 3) {
        build_table(m, c, tab.data());
        build_devconfig(m, c, &dc, &er);
        for (size_t i = 0; i < hull.size(); i++) hull[i] = (&m->foot_hull[0][0][0])[i];   // the model holds real floats
        dc.hull = hull.data();
    }
};
}  // namespace

extern "C" {

// k_dyn over n robots: records [n][96] and targets [n][18] (nullable: zero targets) in, solve records [n][SR_WORDS],
// extension records [n][XR_WORDS] and sort keys [n] out.  Nullable per-robot inputs, as k_dyn reads them:
//   scales [n][4]         friction, servo force limit and servo gain scales (plen_set_env_scales; NULL: all 1)
//   rows   [n][MR_WORDS]  mass rows (plen_set_env_mass): the MASS instance tick_dynamics<true> (NULL: the stock instance)
//   man    [n][PLEN_MAN_WORDS] persistent sole manifolds (config sole_manifold = 1), updated in place as k_dyn does
void emu_dyn(const plen_model *m, const plen_config *c, const float *records, const float *targets, const float *scales,
             const float *rows, float *man, int n, float *srec, float *srx, uint8_t *keys) {
    HostTables T(m, c);
    static WarpScratch ws;
    run_warp([&](int lane) {
        for (int e = 0; e < n; e++) {
            LaneState L;
            load_record(records + 96 * e, ws, L, lane);
            if (lane >= 6 && lane < 24) L.tgt = targets ? targets[18 * e + lane - 6] : 0.0f;
            if (scales) { L.fric_s = scales[4 * e]; L.motor_s = scales[4 * e + 1]; L.kp_s = scales[4 * e + 2]; }
            float *sr = srec + (size_t)e * SR_WORDS, *sx = srx + (size_t)e * XR_WORDS, *mn = man ? man + (size_t)e * PLEN_MAN_WORDS : nullptr;
            if (rows) {
                L.mass_w = rows[(size_t)e * MR_WORDS + lane];
                tick_dynamics<true>(T.dc, T.tab.data(), ws, L, lane, sr, keys + e, nullptr, sx, mn);
            } else {
                tick_dynamics(T.dc, T.tab.data(), ws, L, lane, sr, keys + e, nullptr, sx, mn);
            }
        }
    });
}

// k_solve over given records: groups of PLEN_SOLVE_ROBOTS robots taken from order[0 .. m) in turn (an entry >= n, or a slot
// past m, is an invalid lane; order NULL: robots 0 .. n-1), each through the instance k_rank would route it to: the EXT
// instance iff the group holds a robot with key >= PLEN_KEY_EXT.  records [n][96] are updated in place.
void emu_solve(const plen_model *m, const plen_config *c, float *records, const float *srec, const float *srx, const uint8_t *keys,
               const int *order, int m_order, int n) {
    HostTables T(m, c);
    std::vector<float> Gs(PLEN_SOLVE_ROBOTS * PLEN_GS_WORDS);
    const int len = order ? m_order : n;
    auto robot = [&](int i) { return i >= len ? n : (order ? order[i] : i); };
    run_warp([&](int lane) {
        for (int b = 0; b < len; b += PLEN_SOLVE_ROBOTS) {
            const int r = robot(b + (lane >> 2));
            const bool valid = r >= 0 && r < n;
            const int rr = valid ? r : 0;
            bool anyx = false;
            for (int k = b; k < b + PLEN_SOLVE_ROBOTS; k++) {
                const int q = robot(k);
                anyx = anyx || (q >= 0 && q < n && keys[q] >= PLEN_KEY_EXT);
            }
            if (anyx) {
                const int nx = (valid && keys[rr] >= PLEN_KEY_EXT) ? (int)srx[(size_t)rr * XR_WORDS + XR_NX] : 0;
                solve_tick<1>(T.dc, srec + (size_t)rr * SR_WORDS, Gs.data() + (lane >> 2) * PLEN_GS_WORDS, records + 96 * rr, lane, valid,
                              srx + (size_t)rr * XR_WORDS, nx);
            } else {
                solve_tick<0>(T.dc, srec + (size_t)rr * SR_WORDS, Gs.data() + (lane >> 2) * PLEN_GS_WORDS, records + 96 * rr, lane, valid);
            }
            bar();
        }
    });
}

int emu_sr_words() { return SR_WORDS; }
int emu_xr_words() { return XR_WORDS; }
}
