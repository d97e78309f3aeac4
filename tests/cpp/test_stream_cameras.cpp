// C++ check of per-stream calibration: one dynamic_vins::BatchFeatureTracker serving several rigs, each stream set with
// SetStreamCamera from its own calibration files (dvfe_camera_from_yaml), two frames in flight; writes every stream's records in
// the SerializePointFeature text format, like test_stream_presence.
//   usage: test_stream_cameras <config.yaml> <cams_dir> <frames.bin> <n_frames> <n_streams> <out_prefix> <n_groups>
// cams_dir holds s<stream>_cam0.yaml and s<stream>_cam1.yaml (camodocal PINHOLE) for every stream.
// frames.bin: n_frames x (n_streams x time0 f64, n_streams x gray0, n_streams x gray1)
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "dvfe/feature_tracker.hpp"

static void write_points(const char* prefix, int stream, int k, const dynamic_vins::FeatureBackground& fb) {
    char path[512];
    std::snprintf(path, sizeof(path), "%s_s%d_%d_point.txt", prefix, stream, k);
    std::FILE* fo = std::fopen(path, "w");
    for (const auto& kv : fb.points) {
        std::fprintf(fo, "%d %u", kv.second.size() == 1 ? 0 : 1, kv.first);
        for (const auto& obs : kv.second)
            for (double v : obs.second) std::fprintf(fo, " %.17g", v);
        std::fprintf(fo, "\n");
    }
    std::fclose(fo);
}

static dvfe_camera load_camera(const std::string& path) {
    dvfe_camera c;
    if (dvfe_camera_from_yaml(path.c_str(), &c) != DVFE_OK) throw std::runtime_error(dvfe_last_error(nullptr));
    return c;
}

int main(int argc, char** argv) {
    if (argc < 8) {
        std::fprintf(stderr, "usage: test_stream_cameras <cfg> <cams_dir> <frames> <n_frames> <n_streams> <out> <n_groups>\n");
        return 2;
    }
    try {
        const int n_frames = std::atoi(argv[4]), B = std::atoi(argv[5]), G = std::atoi(argv[7]);
        dynamic_vins::BatchFeatureTracker tracker(argv[1], B, G);
        const int W = tracker.config().width, H = tracker.config().height;
        const size_t P = (size_t)W * H;
        for (int s = 0; s < B; s++) {
            const std::string base = std::string(argv[2]) + "/s" + std::to_string(s);
            const dvfe_camera c0 = load_camera(base + "_cam0.yaml"), c1 = load_camera(base + "_cam1.yaml");
            tracker.SetStreamCamera(s, c0, &c1);
        }
        // a bad calibration and a bad stream index are rejected
        try {
            dvfe_camera bad = load_camera(std::string(argv[2]) + "/s0_cam0.yaml");
            bad.fx = std::nan("");
            tracker.SetStreamCamera(0, bad);
            std::fprintf(stderr, "NaN fx accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("camera value check: ok\n");
        }
        try {
            tracker.SetStreamCamera(B, load_camera(std::string(argv[2]) + "/s0_cam0.yaml"));
            std::fprintf(stderr, "stream index B accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("stream index check: ok\n");
        }
        std::ifstream fin(argv[3], std::ios::binary);
        std::vector<std::vector<uint8_t>> L(n_frames, std::vector<uint8_t>(B * P)), R(n_frames, std::vector<uint8_t>(B * P));
        std::vector<std::vector<double>> T(n_frames, std::vector<double>(B));
        for (int k = 0; k < n_frames; k++) {
            fin.read(reinterpret_cast<char*>(T[k].data()), (std::streamsize)(B * sizeof(double)));
            fin.read(reinterpret_cast<char*>(L[k].data()), (std::streamsize)(B * P));
            fin.read(reinterpret_cast<char*>(R[k].data()), (std::streamsize)(B * P));
        }
        if (!fin) { std::fprintf(stderr, "short frames file\n"); return 2; }
        for (int k = 0; k < n_frames; k++) {
            tracker.TrackImageAsync(L[k].data(), R[k].data(), P, W, T[k]);
            if (k > 0) {
                tracker.Wait();
                for (int s = 0; s < B; s++) write_points(argv[6], s, k - 1, tracker.Features(s));
            }
        }
        tracker.Wait();
        for (int s = 0; s < B; s++) write_points(argv[6], s, n_frames - 1, tracker.Features(s));
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
