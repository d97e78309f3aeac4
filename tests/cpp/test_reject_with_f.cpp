// C++ check of the in-step RejectWithF: dynamic_vins::BatchFeatureTracker (2 streams, 2 stream groups) with
// SetRejectWithF(F_threshold of the settings file, dvfe_f_threshold_from_yaml).  Writes each stream's records of every frame in the
// SerializePointFeature text format; a negative threshold must throw.
//   usage: test_reject_with_f <config.yaml> <frames.bin> <n_frames> <out_prefix>
// frames.bin: n_frames x (2 x time0 f64, 2 x gray0, 2 x gray1)
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "dvfe/feature_tracker.hpp"

static void write_points(const char* prefix, int k, int s, const dynamic_vins::FeatureBackground& fb) {
    char path[512];
    std::snprintf(path, sizeof(path), "%s_%d_%d_point.txt", prefix, k, s);
    std::FILE* fo = std::fopen(path, "w");
    for (const auto& kv : fb.points) {
        std::fprintf(fo, "%d %u", kv.second.size() == 1 ? 0 : 1, kv.first);
        for (const auto& obs : kv.second)
            for (double v : obs.second) std::fprintf(fo, " %.17g", v);
        std::fprintf(fo, "\n");
    }
    std::fclose(fo);
}

int main(int argc, char** argv) {
    if (argc < 5) {
        std::fprintf(stderr, "usage: test_reject_with_f <cfg> <frames> <n_frames> <out>\n");
        return 2;
    }
    try {
        const int n_frames = std::atoi(argv[3]);
        double f = 0.0;
        if (dvfe_f_threshold_from_yaml(argv[1], &f) != DVFE_OK || f <= 0.0) {
            std::fprintf(stderr, "F_threshold: %s\n", dvfe_last_error(nullptr));
            return 1;
        }
        dynamic_vins::BatchFeatureTracker trk(argv[1], 2, 2);
        try {
            trk.SetRejectWithF(-1.0);
            std::fprintf(stderr, "negative threshold accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("negative threshold refused\n");
        }
        trk.SetRejectWithF(f);
        const int W = trk.config().width, H = trk.config().height;
        const size_t P = (size_t)W * H;
        std::ifstream fin(argv[2], std::ios::binary);
        std::vector<uint8_t> L(2 * P), R(2 * P);
        std::vector<double> T(2);
        for (int k = 0; k < n_frames; k++) {
            fin.read(reinterpret_cast<char*>(T.data()), (std::streamsize)(2 * sizeof(double)));
            fin.read(reinterpret_cast<char*>(L.data()), (std::streamsize)(2 * P));
            fin.read(reinterpret_cast<char*>(R.data()), (std::streamsize)(2 * P));
            if (!fin) { std::fprintf(stderr, "short frames file\n"); return 2; }
            trk.TrackImageAsync(L.data(), R.data(), P, W, T);
            trk.Wait();
            for (int s = 0; s < 2; s++) write_points(argv[4], k, s, trk.Features(s));
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
