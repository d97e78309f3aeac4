// C++ check of stream snapshots: stream 1 of one dynamic_vins::BatchFeatureTracker (2 streams) is moved with ExportStream /
// ImportStream to slot 2 of another (3 streams, 2 stream groups, no frame yet) after k0 frames and continues there; a truncated blob
// is refused.  Writes the moved stream's records of frames k0.. in the SerializePointFeature text format, like test_stream_presence.
//   usage: test_stream_snapshot <config.yaml> <frames.bin> <n_frames> <k0> <out_prefix>
// frames.bin: n_frames x (2 x time0 f64, 2 x gray0, 2 x gray1)
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "dvfe/feature_tracker.hpp"

static void write_points(const char* prefix, int k, const dynamic_vins::FeatureBackground& fb) {
    char path[512];
    std::snprintf(path, sizeof(path), "%s_%d_point.txt", prefix, k);
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
    if (argc < 6) {
        std::fprintf(stderr, "usage: test_stream_snapshot <cfg> <frames> <n_frames> <k0> <out>\n");
        return 2;
    }
    try {
        const int n_frames = std::atoi(argv[3]), k0 = std::atoi(argv[4]);
        dynamic_vins::BatchFeatureTracker src(argv[1], 2, 1);
        dynamic_vins::BatchFeatureTracker dst(argv[1], 3, 2);
        const int W = src.config().width, H = src.config().height;
        const size_t P = (size_t)W * H;
        std::ifstream fin(argv[2], std::ios::binary);
        std::vector<std::vector<uint8_t>> L(n_frames, std::vector<uint8_t>(2 * P)), R(n_frames, std::vector<uint8_t>(2 * P));
        std::vector<std::vector<double>> T(n_frames, std::vector<double>(2));
        for (int k = 0; k < n_frames; k++) {
            fin.read(reinterpret_cast<char*>(T[k].data()), (std::streamsize)(2 * sizeof(double)));
            fin.read(reinterpret_cast<char*>(L[k].data()), (std::streamsize)(2 * P));
            fin.read(reinterpret_cast<char*>(R[k].data()), (std::streamsize)(2 * P));
        }
        if (!fin) { std::fprintf(stderr, "short frames file\n"); return 2; }
        for (int k = 0; k < k0; k++) {
            src.TrackImageAsync(L[k].data(), R[k].data(), P, W, T[k]);
            src.Wait();
        }
        const std::vector<uint8_t> blob = src.ExportStream(1);
        try {
            dst.ImportStream(2, std::vector<uint8_t>(blob.begin(), blob.end() - 1));
            std::fprintf(stderr, "truncated blob accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("truncated blob check: ok\n");
        }
        dst.ImportStream(2, blob);
        // every slot of the destination gets the moved stream's frame; slots 0 and 1 start their own tracks with it
        std::vector<uint8_t> l(3 * P), r(3 * P);
        for (int k = k0; k < n_frames; k++) {
            for (int s = 0; s < 3; s++) {
                std::copy(L[k].begin() + P, L[k].end(), l.begin() + s * P);
                std::copy(R[k].begin() + P, R[k].end(), r.begin() + s * P);
            }
            dst.TrackImageAsync(l.data(), r.data(), P, W, std::vector<double>(3, T[k][1]));
            dst.Wait();
            write_points(argv[5], k, dst.Features(2));
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
