// host_shim_reanchor_test.cpp -- re-anchoring through myslam::DeviceOdometry: step() through every rotation but the last,
// detectLoop() with loopParams().min_gap = min_gap, trajectory(), reanchor() to that trajectory with update u shifted by
// 10 u mm along x (the stand-in for a pose-graph back end), then step() on the last rotation and trajectory() again.
// Writes accepted (int32), the pose reanchor() set, the last step's pose and the final trajectory (row-major 4x4 float32);
// tests/test_reanchor.py compares them with the Python calls.
// usage: host_shim_reanchor_test ring.bin out.bin min_gap rot0.bin rot1.bin [rot2.bin ...]
//   ring.bin: float64 vertical angles; rot*.bin: n records {float64 azimuth, float64 vertical, uint16 distance}
// Exits 1 with the library's message when no usable GPU (or any other error) is there.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <vector>

#include "../b-shot-slam_b200/host/device_odometry.h"

static std::vector<char> slurp(const char* path) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    const std::streamsize bytes = f.tellg();
    std::vector<char> raw(bytes > 0 ? (size_t)bytes : 0);
    f.seekg(0);
    if (bytes > 0) f.read(raw.data(), bytes);
    return raw;
}

static std::vector<velodyne::Laser> read_lasers(const char* path) {
    const std::vector<char> raw = slurp(path);
    const size_t rec = 8 + 8 + 2, n = raw.size() / rec;
    std::vector<velodyne::Laser> lasers(n);
    for (size_t i = 0; i < n; ++i) {
        std::memcpy(&lasers[i].azimuth, &raw[rec * i], 8);
        std::memcpy(&lasers[i].vertical, &raw[rec * i + 8], 8);
        std::memcpy(&lasers[i].distance, &raw[rec * i + 16], 2);
    }
    return lasers;
}

static void write_pose(std::ofstream& out, const Matrix4f& T) {
    float rm[16];
    for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) rm[4 * r + c] = T(r, c);
    out.write(reinterpret_cast<const char*>(rm), sizeof(rm));
}

int main(int argc, char** argv) {
    if (argc < 6) return 2;
    myslam::DeviceOdometry odo;
    if (odo.last_status() != BSHOT_OK) { std::printf("context: %s\n", bshot_last_error()); return 1; }
    const std::vector<char> rb = slurp(argv[1]);
    std::vector<double> ring(rb.size() / 8);
    std::memcpy(ring.data(), rb.data(), 8 * ring.size());
    for (int k = 4; k < argc - 1; ++k) {
        odo.step(read_lasers(argv[k]), ring);
        if (odo.last_status() != BSHOT_OK) { std::printf("step %d: %s\n", k - 4, bshot_last_error()); return 1; }
    }
    odo.loopParams().min_gap = std::atoi(argv[3]);
    bshot_loop_report r = bshot_loop_report();
    const int accepted = odo.detectLoop(&r) ? 1 : 0;
    if (odo.last_status() != BSHOT_OK) { std::printf("detectLoop: %s\n", bshot_last_error()); return 1; }
    std::vector<Matrix4f> traj;
    odo.trajectory(traj);
    if (odo.last_status() != BSHOT_OK) { std::printf("trajectory: %s\n", bshot_last_error()); return 1; }
    for (size_t u = 0; u < traj.size(); ++u) traj[u](0, 3) += 10.0f * (float)u;
    if (odo.reanchor(traj) != BSHOT_OK) { std::printf("reanchor: %s\n", bshot_last_error()); return 1; }
    const Matrix4f anchored = odo.pose();
    const Matrix4f last = odo.step(read_lasers(argv[argc - 1]), ring);
    if (odo.last_status() != BSHOT_OK) { std::printf("last step: %s\n", bshot_last_error()); return 1; }
    odo.trajectory(traj);
    if (odo.last_status() != BSHOT_OK) { std::printf("trajectory: %s\n", bshot_last_error()); return 1; }
    std::ofstream out(argv[2], std::ios::binary);
    out.write(reinterpret_cast<const char*>(&accepted), sizeof(accepted));
    write_pose(out, anchored);
    write_pose(out, last);
    for (const Matrix4f& T : traj) write_pose(out, T);
    std::printf("scan %d: accepted %d, match %d; re-anchored pose t = (%.1f, %.1f, %.1f); %zu poses\n", r.scan, accepted, r.match_scan, anchored(0, 3),
                anchored(1, 3), anchored(2, 3), traj.size());
    return 0;
}
