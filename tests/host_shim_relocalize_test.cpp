// host_shim_relocalize_test.cpp -- save a map, restore it elsewhere and find a rotation in it with myslam::DeviceOdometry:
// odometry A steps through the mapping rotations, exportMap -> importMap into a fresh odometry B, B.relocalize(query
// rotation), then B.step(next rotation).  Writes B's relocalised pose and step pose (row-major 4x4, float32) and a few
// report fields; tests/test_relocalize.py compares them with the Python calls.
// usage: host_shim_relocalize_test ring.bin out.bin query.bin next.bin map0.bin [map1.bin ...]
//   ring.bin: float64 vertical angles; *.bin: n records {float64 azimuth, float64 vertical, uint16 distance}
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
    myslam::DeviceOdometry a, b;
    if (a.last_status() != BSHOT_OK || b.last_status() != BSHOT_OK) { std::printf("context: %s\n", bshot_last_error()); return 1; }
    const std::vector<char> rb = slurp(argv[1]);
    std::vector<double> ring(rb.size() / 8);
    std::memcpy(ring.data(), rb.data(), 8 * ring.size());
    for (int k = 5; k < argc; ++k) {
        a.step(read_lasers(argv[k]), ring);
        if (a.last_status() != BSHOT_OK) { std::printf("map step %d: %s\n", k - 5, bshot_last_error()); return 1; }
    }
    std::vector<float> xyzr;
    std::vector<bshot_descriptor> desc;
    if (a.exportMap(xyzr, desc) != BSHOT_OK) { std::printf("export: %s\n", bshot_last_error()); return 1; }
    if (b.importMap(xyzr, desc) != BSHOT_OK) { std::printf("import: %s\n", bshot_last_error()); return 1; }
    const bool accepted = b.relocalize(read_lasers(argv[3]), ring);
    if (b.last_status() != BSHOT_OK) { std::printf("relocalize: %s\n", bshot_last_error()); return 1; }
    std::ofstream out(argv[2], std::ios::binary);
    const bshot_reloc_report& r = b.reloc_report();
    out.write(reinterpret_cast<const char*>(r.pose), sizeof(r.pose));
    const int fields[5] = {(int)desc.size(), r.n_keypoints, r.n_pairs, r.n_inliers, r.accepted};
    out.write(reinterpret_cast<const char*>(fields), sizeof(fields));
    std::printf("map %zu entries; relocalised: accepted %d, %d inliers, t = (%.1f, %.1f, %.1f)\n", desc.size(), (int)accepted, r.n_inliers, r.pose[3],
                r.pose[7], r.pose[11]);
    const Matrix4f T = b.step(read_lasers(argv[4]), ring);
    if (b.last_status() != BSHOT_OK) { std::printf("step: %s\n", bshot_last_error()); return 1; }
    write_pose(out, T);
    return 0;
}
