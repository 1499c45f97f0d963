// TEST-ONLY warp emulation of the per-robot reset settle (plen_settle_env_resets).  Builds on the harness of emu_warp.cpp (the
// product's device source compiled for the host) and exports start_record, the device function k_start_records applies to
// each robot's (x, y, z, yaw), in the precision of the build.  The settle ticks themselves are emu_warp.cpp's emu_tick with
// zero targets, as launch_ticks runs them.  Never linked into the product library.
#include "emu_warp.cpp"

extern "C" {
// pose [4] = x, y, z, yaw -> rec [96]
void emu_start_record(const float *pose, float *rec) { start_record(pose[0], pose[1], pose[2], pose[3], rec); }
}
