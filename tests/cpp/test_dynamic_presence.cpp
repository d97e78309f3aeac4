// C++ check of per-stream frame presence in dynamic mode: drives dynamic_vins::BatchFeatureTracker::TrackDynamicAsync(...,
// stream_flags) with two frames in flight and writes every stream's background and instance records in the formats of
// test_feature_tracker dynbatch.
//   usage: test_dynamic_presence <config.yaml> <frames.bin> <n_frames> <n_streams> <out_prefix> <n_groups> <max_instances>
// frames.bin: n_frames x (n_streams flag bytes, then n_streams records of test_feature_tracker's dynamic frame layout:
//   time0 f64, gray0, gray1, inv_merge_mask (H*W each), exist i32, n_boxes i32, n_boxes x (track_id, x, y, w, h i32, mask w*h))
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "dvfe/feature_tracker.hpp"

namespace {

struct Frame {
    double time0 = 0;
    int exist = 0;
    std::vector<std::vector<uint8_t>> masks;
    std::vector<dynamic_vins::Box2D::Ptr> boxes;
};

void read_frame(std::ifstream& fin, size_t P, Frame& f, uint8_t* g0, uint8_t* g1, uint8_t* inv) {
    fin.read(reinterpret_cast<char*>(&f.time0), sizeof(double));
    fin.read(reinterpret_cast<char*>(g0), (std::streamsize)P);
    fin.read(reinterpret_cast<char*>(g1), (std::streamsize)P);
    fin.read(reinterpret_cast<char*>(inv), (std::streamsize)P);
    int n = 0;
    fin.read(reinterpret_cast<char*>(&f.exist), 4);
    fin.read(reinterpret_cast<char*>(&n), 4);
    f.masks.resize(n);
    for (int b = 0; b < n; b++) {
        int v[5];
        fin.read(reinterpret_cast<char*>(v), 20);
        f.masks[b].resize((size_t)v[3] * v[4]);
        fin.read(reinterpret_cast<char*>(f.masks[b].data()), (std::streamsize)f.masks[b].size());
        auto box = std::make_shared<dynamic_vins::Box2D>();
        box->track_id = v[0]; box->id = b;
        box->rect = {(float)v[1], (float)v[2], (float)v[3], (float)v[4]};
        box->min_pt = {(float)v[1], (float)v[2]};
        box->max_pt = {(float)(v[1] + v[3]), (float)(v[2] + v[4])};
        box->roi = std::make_shared<dynamic_vins::InstRoi>();
        box->roi->mask_cv = {f.masks[b].data(), v[4], v[3], v[3]};
        f.boxes.push_back(box);
    }
}

void write_points(const char* prefix, int stream, int k, const dynamic_vins::FeatureBackground& fb) {
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

void write_instances(const char* prefix, int stream, int k, const std::map<unsigned int, dynamic_vins::FeatureInstance>& insts) {
    char path[512];
    std::snprintf(path, sizeof(path), "%s_s%d_%d_inst.txt", prefix, stream, k);
    std::FILE* fo = std::fopen(path, "w");
    for (const auto& kv : insts)
        for (const auto& fp : kv.second.features) {
            const dynamic_vins::FeaturePoint& f = *fp.second;
            std::fprintf(fo, "%u %u %d %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.9g %d\n", kv.first, fp.first,
                         f.is_stereo ? 1 : 0, f.point[0], f.point[1], f.point[2], f.vel[0], f.vel[1], f.point_right[0],
                         f.point_right[1], f.point_right[2], f.vel_right[0], f.vel_right[1], (double)f.disp, -1);
        }
    std::fclose(fo);
}

}  // namespace

int main(int argc, char** argv) {
    if (argc < 8) {
        std::fprintf(stderr, "usage: test_dynamic_presence <cfg> <frames> <n_frames> <n_streams> <out> <n_groups> <max_instances>\n");
        return 2;
    }
    try {
        const int n_frames = std::atoi(argv[3]), B = std::atoi(argv[4]), G = std::atoi(argv[6]);
        dynamic_vins::BatchFeatureTracker tracker(argv[1], B, G, std::atoi(argv[7]));
        const int W = tracker.config().width, H = tracker.config().height;
        const size_t P = (size_t)W * H;
        std::ifstream fin(argv[2], std::ios::binary);
        std::vector<std::vector<uint8_t>> F(n_frames, std::vector<uint8_t>(B));
        std::vector<std::vector<uint8_t>> L(n_frames, std::vector<uint8_t>(B * P)), R(n_frames, std::vector<uint8_t>(B * P)),
            M(n_frames, std::vector<uint8_t>(B * P));
        std::vector<std::vector<Frame>> D(n_frames, std::vector<Frame>(B));
        for (int k = 0; k < n_frames; k++) {
            fin.read(reinterpret_cast<char*>(F[k].data()), (std::streamsize)B);
            for (int s = 0; s < B; s++) read_frame(fin, P, D[k][s], &L[k][s * P], &R[k][s * P], &M[k][s * P]);
        }
        if (!fin) { std::fprintf(stderr, "short frames file\n"); return 2; }
        auto enqueue = [&](int k, const std::vector<uint8_t>& flags) {
            std::vector<int> exist(B);
            std::vector<std::vector<dynamic_vins::Box2D::Ptr>> boxes(B);
            std::vector<double> t(B);
            for (int s = 0; s < B; s++) { exist[s] = D[k][s].exist; boxes[s] = D[k][s].boxes; t[s] = D[k][s].time0; }
            tracker.TrackDynamicAsync(L[k].data(), R[k].data(), M[k].data(), P, W, exist, boxes, t, flags);
        };
        // a flag vector of the wrong length is rejected before anything is enqueued
        try {
            enqueue(0, std::vector<uint8_t>(B + 1, 0));
            std::fprintf(stderr, "wrong flag length accepted\n");
            return 1;
        } catch (const std::runtime_error&) {
            std::printf("flag length check: ok\n");
        }
        for (int k = 0; k < n_frames; k++) {
            enqueue(k, F[k]);
            if (k > 0) {
                tracker.Wait();
                for (int s = 0; s < B; s++) { write_points(argv[5], s, k - 1, tracker.Features(s)); write_instances(argv[5], s, k - 1, tracker.InstsOutput(s)); }
            }
        }
        tracker.Wait();
        for (int s = 0; s < B; s++) { write_points(argv[5], s, n_frames - 1, tracker.Features(s)); write_instances(argv[5], s, n_frames - 1, tracker.InstsOutput(s)); }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
