// host_shim_voxel_test.cpp -- drives the reference-named `bshot` shim through voxel-grid keypoints:
// cloud1 / cloud2 <- two clouds read from raw float32 xyz files, calculate_voxel_grid_keypoints(leaf), then
// calculate_normals(3000) -> calculate_SHOT(3000) -> compute_bshot() on cloud1's voxel keypoints.  Writes
// cloud1_keypoints, cloud2_keypoints (count + xyz each, with width / height / is_dense) and the B-SHOT bits;
// tests/test_voxel_grid.py checks them against the Python path.
// usage: host_shim_voxel_test cloud1.bin cloud2.bin leaf out.bin [organize]
// `organize` gives both clouds an organized layout (height 2, is_dense false) and stops after the keypoints: the output
// clouds then show whether the shim took PCL's overflow copy (the input's layout) or binned (width = count, height 1).
#include <cstdio>
#include <cstdlib>
#include <fstream>

#include "../b-shot-slam_b200/host/bshot_bits.h"

static void load(const char* path, pcl::PointCloud<pcl::PointXYZ>& pc) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    const size_t bytes = (size_t)f.tellg();
    f.seekg(0);
    std::vector<float> raw(bytes / 4);
    f.read(reinterpret_cast<char*>(raw.data()), (std::streamsize)bytes);
    pc.clear();
    for (size_t i = 0; i + 2 < raw.size(); i += 3) pc.push_back(pcl::PointXYZ(raw[i], raw[i + 1], raw[i + 2]));
}

static void write_cloud(std::ofstream& out, const pcl::PointCloud<pcl::PointXYZ>& pc) {
    const int hdr[4] = {(int)pc.size(), (int)pc.width, (int)pc.height, (int)pc.is_dense};
    out.write(reinterpret_cast<const char*>(hdr), sizeof(hdr));
    for (const auto& p : pc.points) out.write(reinterpret_cast<const char*>(p.data), 12);
}

int main(int argc, char** argv) {
    if (argc < 5) return 2;
    bshot cb(0, 1u << 18, 1u << 14, 1u << 10);
    if (cb.last_status() != BSHOT_OK) { std::printf("ctx: %s\n", bshot_last_error()); return 1; }
    load(argv[1], cb.cloud1);
    load(argv[2], cb.cloud2);
    const bool organize = argc > 5 && std::string(argv[5]) == "organize";
    if (organize)
        for (auto* pc : {&cb.cloud1, &cb.cloud2}) { pc->width = (uint32_t)(pc->size() / 2); pc->height = 2; pc->is_dense = false; }
    cb.calculate_voxel_grid_keypoints((float)std::atof(argv[3]));
    if (cb.last_status() != BSHOT_OK) { std::printf("voxel grid: %s\n", bshot_last_error()); return 1; }
    std::ofstream out(argv[4], std::ios::binary);
    write_cloud(out, cb.cloud1_keypoints);
    write_cloud(out, cb.cloud2_keypoints);
    if (organize) return 0;
    cb.calculate_normals(3000);
    cb.calculate_SHOT(3000);
    cb.compute_bshot();
    if (cb.last_status() != BSHOT_OK) { std::printf("descriptors: %s\n", bshot_last_error()); return 1; }
    const int nb = (int)cb.cloud1_bshot.size();
    out.write(reinterpret_cast<const char*>(&nb), 4);
    out.write(reinterpret_cast<const char*>(cb.cloud1_bshot.data()), 48 * (size_t)nb);
    std::printf("voxel keypoints: %zu / %zu, descriptors %d\n", cb.cloud1_keypoints.size(), cb.cloud2_keypoints.size(), nb);
    return 0;
}
