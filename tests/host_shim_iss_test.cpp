// host_shim_iss_test.cpp -- drives the reference-named C++ shims in the call order of the reference's kp_test driver
// (setSrcFrame -> extractKeypoints -> issKpDetection -> computeDescriptors -> featureMatching -> evaluateEstimation ->
// poseEstimation -> updateMap -> kpEvaluation) over two clouds read from raw float32 xyz files.  Writes per frame the
// seg-ratio and ISS keypoints, the pose and the two repeat rates; tests/test_iss.py checks them against the Python path.
// usage: host_shim_iss_test cloud0.bin cloud1.bin out.bin
#include <cstdio>
#include <fstream>

#include "../b-shot-slam_b200/host/lidar_odometry.h"

static myslam::Frame::PCPtr load(const char* path) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    const size_t bytes = (size_t)f.tellg();
    f.seekg(0);
    std::vector<float> raw(bytes / 4);
    f.read(reinterpret_cast<char*>(raw.data()), (std::streamsize)bytes);
    auto pc = std::make_shared<std::vector<Vector3f>>();
    for (size_t i = 0; i + 2 < raw.size(); i += 3) pc->push_back(Vector3f(raw[i], raw[i + 1], raw[i + 2]));
    return pc;
}

int main(int argc, char** argv) {
    if (argc < 4) return 2;
    myslam::LidarOdometry lo(0);
    if (lo.last_status() != BSHOT_OK) { std::printf("ctx: %s\n", bshot_last_error()); return 1; }
    std::ofstream out(argv[3], std::ios::binary);
    for (int fidx = 0; fidx < 2; ++fidx) {
        myslam::Frame::Ptr f = myslam::Frame::createFrame();
        f->setPointCloud(load(argv[1 + fidx]));
        if (fidx > 0) lo.passSrc2Ref();
        lo.setSrcFrame(f);
        lo.extractKeypoints();
        lo.issKpDetection();
        lo.computeDescriptors();
        lo.featureMatching();
        lo.evaluateEstimation();
        lo.poseEstimation();
        lo.updateMap();
        lo.kpEvaluation();
        if (lo.last_status() != BSHOT_OK) { std::printf("frame %d: %s\n", fidx, bshot_last_error()); return 1; }
        const int nk = (int)f->getKeypoints()->size(), ni = (int)f->getISSKeypoints()->size();
        out.write(reinterpret_cast<const char*>(&nk), 4);
        out.write(reinterpret_cast<const char*>(&ni), 4);
        for (auto& p : *f->getKeypoints()) out.write(reinterpret_cast<const char*>(p.v), 12);
        for (auto& p : *f->getISSKeypoints()) out.write(reinterpret_cast<const char*>(p.v), 12);
        float T[16];
        myslam::LidarOdometry::to_row_major(f->getPose(), T);
        out.write(reinterpret_cast<const char*>(T), 64);
        out.write(reinterpret_cast<const char*>(&lo.sr_repeat_rate_), 8);
        out.write(reinterpret_cast<const char*>(&lo.iss_repeat_rate_), 8);
        std::printf("frame %d: %d seg-ratio keypoints, %d ISS keypoints, repeat rate %.4f / %.4f\n", fidx, nk, ni, lo.sr_repeat_rate_,
                    lo.iss_repeat_rate_);
    }
    return 0;
}
