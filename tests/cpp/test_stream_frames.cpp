// C++ check of per-camera frame descriptors: drives dynamic_vins::BatchFeatureTracker::TrackFramesAsync over one
// std::vector<uint8_t> per camera image, each with its own row pitch, with two frames in flight, and writes every stream's
// records in the SerializePointFeature text format, like test_stream_presence.
//   usage: test_stream_frames <config.yaml> <frames.bin> <n_frames> <n_streams> <out_prefix> <n_groups>
// frames.bin: n_frames x n_streams x (flags u8: 1 = no frame, 2 = no right image, 4 = reset; time0 f64; pitch i32;
//             then the left image, and the right image unless flag 2, of H rows of `pitch` bytes each; nothing when flag 1)
#include <cstdint>
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

struct Camera {                        // one camera's buffers of one frame, as a decoder would hand them over
    uint8_t flags = 0;
    double time0 = 0.0;
    int32_t pitch = 0;
    std::vector<uint8_t> left, right;
};

int main(int argc, char** argv) {
    if (argc < 7) { std::fprintf(stderr, "usage: test_stream_frames <cfg> <frames> <n_frames> <n_streams> <out> <n_groups>\n"); return 2; }
    try {
        const int n_frames = std::atoi(argv[3]), B = std::atoi(argv[4]), G = std::atoi(argv[6]);
        dynamic_vins::BatchFeatureTracker tracker(argv[1], B, G);
        const int H = tracker.config().height;
        std::ifstream fin(argv[2], std::ios::binary);
        std::vector<std::vector<Camera>> cams(n_frames, std::vector<Camera>(B));
        for (int k = 0; k < n_frames; k++)
            for (int s = 0; s < B; s++) {
                Camera& c = cams[k][s];
                fin.read(reinterpret_cast<char*>(&c.flags), 1);
                fin.read(reinterpret_cast<char*>(&c.time0), sizeof(double));
                fin.read(reinterpret_cast<char*>(&c.pitch), sizeof(int32_t));
                if (c.flags & 1) continue;
                c.left.resize((size_t)H * c.pitch);
                fin.read(reinterpret_cast<char*>(c.left.data()), (std::streamsize)c.left.size());
                if (c.flags & 2) continue;
                c.right.resize((size_t)H * c.pitch);
                fin.read(reinterpret_cast<char*>(c.right.data()), (std::streamsize)c.right.size());
            }
        if (!fin) { std::fprintf(stderr, "short frames file\n"); return 2; }
        auto describe = [&](int k) {
            std::vector<dvfe_frame> d(B);
            for (int s = 0; s < B; s++) {
                const Camera& c = cams[k][s];
                d[s] = dvfe_frame{};
                d[s].left = c.left.empty() ? nullptr : c.left.data();
                d[s].right = c.right.empty() ? nullptr : c.right.data();
                d[s].pitch = c.pitch;
                d[s].flags = (c.flags & 4) ? DVFE_FRAME_RESET : 0u;
                d[s].time0 = c.time0;
            }
            return d;
        };
        // a descriptor array of the wrong length, and a restart without a frame, are rejected before anything is enqueued
        try {
            tracker.TrackFramesAsync(std::vector<dvfe_frame>(B + 1));
            std::fprintf(stderr, "wrong descriptor count accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("frame count check: ok\n");
        }
        try {
            std::vector<dvfe_frame> bad = describe(0);
            bad[0].left = nullptr;
            bad[0].flags = DVFE_FRAME_RESET;
            tracker.TrackFramesAsync(bad);
            std::fprintf(stderr, "RESET without a frame accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("frame value check: ok\n");
        }
        for (int k = 0; k < n_frames; k++) {
            tracker.TrackFramesAsync(describe(k));
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
