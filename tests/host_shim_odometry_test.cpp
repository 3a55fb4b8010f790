// host_shim_odometry_test.cpp -- drives myslam::DeviceOdometry the way odometry_test.cpp's loop would: every rotation read
// from a raw file becomes a std::vector<velodyne::Laser>, and one step() call per rotation returns the pose.  Writes the
// row-major 4x4 poses (float32) and a few report fields; tests/test_odometry_step.py compares them with the Python step.
// usage: host_shim_odometry_test ring.bin out.bin rot0.bin [rot1.bin ...]
//   ring.bin: float64 vertical angles; rotN.bin: n records {float64 azimuth, float64 vertical, uint16 distance}
// Exits 1 with the library's message when no usable GPU (or any other error) is there.
#include <cstdio>
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

int main(int argc, char** argv) {
    if (argc < 4) return 2;
    myslam::DeviceOdometry odo;
    if (odo.last_status() != BSHOT_OK) { std::printf("context: %s\n", bshot_last_error()); return 1; }
    const std::vector<char> rb = slurp(argv[1]);
    std::vector<double> ring(rb.size() / 8);
    std::memcpy(ring.data(), rb.data(), 8 * ring.size());
    std::ofstream out(argv[2], std::ios::binary);
    for (int a = 3; a < argc; ++a) {
        const std::vector<char> raw = slurp(argv[a]);
        const size_t rec = 8 + 8 + 2, n = raw.size() / rec;
        std::vector<velodyne::Laser> lasers(n);
        for (size_t i = 0; i < n; ++i) {
            std::memcpy(&lasers[i].azimuth, &raw[rec * i], 8);
            std::memcpy(&lasers[i].vertical, &raw[rec * i + 8], 8);
            std::memcpy(&lasers[i].distance, &raw[rec * i + 16], 2);
        }
        const Matrix4f T = odo.step(lasers, ring);
        if (odo.last_status() != BSHOT_OK) { std::printf("step %d: %s\n", a - 3, bshot_last_error()); return 1; }
        float rm[16];
        for (int r = 0; r < 4; ++r) for (int c = 0; c < 4; ++c) rm[4 * r + c] = T(r, c);
        out.write(reinterpret_cast<const char*>(rm), sizeof(rm));
        const int fields[4] = {odo.report().n_keypoints, odo.report().n_pairs, odo.report().n_inliers, odo.report().was_initial};
        out.write(reinterpret_cast<const char*>(fields), sizeof(fields));
        std::printf("step %d: %d keypoints, %d pairs, %d inliers, t = (%.1f, %.1f, %.1f)\n", a - 3, fields[0], fields[1], fields[2], rm[3], rm[7], rm[11]);
    }
    if (odo.reset() != BSHOT_OK) { std::printf("reset: %s\n", bshot_last_error()); return 1; }
    return 0;
}
