// C++ check of per-stream frame presence: drives dynamic_vins::BatchFeatureTracker::TrackImageAsync(..., stream_flags) with two
// frames in flight and writes every stream's records in the SerializePointFeature text format, like test_feature_tracker batch.
//   usage: test_stream_presence <config.yaml> <frames.bin> <n_frames> <n_streams> <out_prefix> <n_groups>
// frames.bin: n_frames x (n_streams flag bytes, n_streams x time0 f64, n_streams x gray0, n_streams x gray1)
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

int main(int argc, char** argv) {
    if (argc < 7) { std::fprintf(stderr, "usage: test_stream_presence <cfg> <frames> <n_frames> <n_streams> <out> <n_groups>\n"); return 2; }
    try {
        const int n_frames = std::atoi(argv[3]), B = std::atoi(argv[4]), G = std::atoi(argv[6]);
        dynamic_vins::BatchFeatureTracker tracker(argv[1], B, G);
        const int W = tracker.config().width, H = tracker.config().height;
        const size_t P = (size_t)W * H;
        std::ifstream fin(argv[2], std::ios::binary);
        std::vector<std::vector<uint8_t>> F(n_frames, std::vector<uint8_t>(B));
        std::vector<std::vector<uint8_t>> L(n_frames, std::vector<uint8_t>(B * P)), R(n_frames, std::vector<uint8_t>(B * P));
        std::vector<std::vector<double>> T(n_frames, std::vector<double>(B));
        for (int k = 0; k < n_frames; k++) {
            fin.read(reinterpret_cast<char*>(F[k].data()), (std::streamsize)B);
            fin.read(reinterpret_cast<char*>(T[k].data()), (std::streamsize)(B * sizeof(double)));
            fin.read(reinterpret_cast<char*>(L[k].data()), (std::streamsize)(B * P));
            fin.read(reinterpret_cast<char*>(R[k].data()), (std::streamsize)(B * P));
        }
        if (!fin) { std::fprintf(stderr, "short frames file\n"); return 2; }
        // a flag vector of the wrong length and an invalid flag are rejected before anything is enqueued
        try {
            tracker.TrackImageAsync(L[0].data(), R[0].data(), P, W, T[0], std::vector<uint8_t>(B + 1, 0));
            std::fprintf(stderr, "wrong flag length accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("flag length check: ok\n");
        }
        try {
            std::vector<uint8_t> bad(B, 0);
            bad[0] = DVFE_FRAME_SKIP | DVFE_FRAME_RESET;
            tracker.TrackImageAsync(L[0].data(), R[0].data(), P, W, T[0], bad);
            std::fprintf(stderr, "SKIP|RESET accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("flag value check: ok\n");
        }
        for (int k = 0; k < n_frames; k++) {
            tracker.TrackImageAsync(L[k].data(), R[k].data(), P, W, T[k], F[k]);
            if (k > 0) {
                tracker.Wait();
                for (int s = 0; s < B; s++) write_points(argv[5], s, k - 1, tracker.Features(s));
            }
        }
        tracker.Wait();
        for (int s = 0; s < B; s++) write_points(argv[5], s, n_frames - 1, tracker.Features(s));
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
