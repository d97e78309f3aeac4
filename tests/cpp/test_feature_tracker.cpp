// C++ drop-in check: drives include/dvfe/feature_tracker.hpp (the reference-shaped C++ API) exactly like
// FeatureTrack() in dynamic_vins/src/system/main.cpp:178-330 does, on frames dumped by the python test, and writes the
// features in the reference's SerializePointFeature text format (utils/io/feature_serialization.cpp:26-38).
//   usage: test_feature_tracker <config.yaml> <frames.bin> <n_frames> <stereo 0|1> <out_prefix>
// frames.bin: n_frames x (time0 f64, gray0 H*W, [gray1 H*W])
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <fstream>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "dvfe/feature_tracker.hpp"

static void write_points(const char* prefix, int stream, int k, const dynamic_vins::FeatureBackground& fb) {
    char path[512];
    if (stream < 0) std::snprintf(path, sizeof(path), "%s_%d_point.txt", prefix, k);
    else std::snprintf(path, sizeof(path), "%s_s%d_%d_point.txt", prefix, stream, k);
    std::FILE* fo = std::fopen(path, "w");
    for (const auto& kv : fb.points) {
        std::fprintf(fo, "%d %u", kv.second.size() == 1 ? 0 : 1, kv.first);
        for (const auto& obs : kv.second)
            for (double v : obs.second) std::fprintf(fo, " %.17g", v);
        std::fprintf(fo, "\n");
    }
    std::fclose(fo);
}

// batch mode: test_feature_tracker batch <config.yaml> <frames.bin> <n_frames> <n_streams> <out_prefix> <n_groups>
// frames.bin: n_frames x (n_streams x time0 f64, n_streams x gray0, n_streams x gray1); pipelined (two frames in flight)
static int run_batch(int argc, char** argv) {
    if (argc < 8) { std::fprintf(stderr, "usage (batch)\n"); return 2; }
    const int n_frames = std::atoi(argv[4]), B = std::atoi(argv[5]), G = std::atoi(argv[7]);
    dynamic_vins::BatchFeatureTracker tracker(argv[2], B, G);
    const int W = tracker.config().width, H = tracker.config().height;
    const size_t P = (size_t)W * H;
    std::ifstream fin(argv[3], std::ios::binary);
    // the frames of both in-flight steps must stay valid: keep them all
    std::vector<std::vector<uint8_t>> L(n_frames, std::vector<uint8_t>(B * P)), R(n_frames, std::vector<uint8_t>(B * P));
    std::vector<std::vector<double>> T(n_frames, std::vector<double>(B));
    for (int k = 0; k < n_frames; k++) {
        fin.read(reinterpret_cast<char*>(T[k].data()), (std::streamsize)(B * sizeof(double)));
        fin.read(reinterpret_cast<char*>(L[k].data()), (std::streamsize)(B * P));
        fin.read(reinterpret_cast<char*>(R[k].data()), (std::streamsize)(B * P));
    }
    for (int k = 0; k < n_frames; k++) {
        tracker.TrackImageAsync(L[k].data(), R[k].data(), P, W, T[k]);
        if (k > 0) {
            tracker.Wait();
            for (int s = 0; s < B; s++) write_points(argv[6], s, k - 1, tracker.Features(s));
        }
    }
    tracker.Wait();
    for (int s = 0; s < B; s++) write_points(argv[6], s, n_frames - 1, tracker.Features(s));
    return 0;
}

// ---- dynamic mode ------------------------------------------------------------------------------------------------------
// one frame of one stream in frames.bin: time0 f64, gray0 H*W, gray1 H*W, inv_merge_mask H*W, exist_inst i32, n_boxes i32,
// then per box: track_id, x, y, w, h (i32) and the w*h mask bytes
struct DynFrame {
    double time0 = 0;
    std::vector<uint8_t> g0, g1, inv;
    int exist = 0;
    std::vector<std::vector<uint8_t>> masks;
    std::vector<dynamic_vins::Box2D::Ptr> boxes;
};

static void read_dyn_frame(std::ifstream& fin, size_t P, DynFrame& f) {
    f.g0.resize(P); f.g1.resize(P); f.inv.resize(P);
    fin.read(reinterpret_cast<char*>(&f.time0), sizeof(double));
    fin.read(reinterpret_cast<char*>(f.g0.data()), (std::streamsize)P);
    fin.read(reinterpret_cast<char*>(f.g1.data()), (std::streamsize)P);
    fin.read(reinterpret_cast<char*>(f.inv.data()), (std::streamsize)P);
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

static void write_instances(const char* prefix, int stream, int k, const std::map<unsigned int, dynamic_vins::FeatureInstance>& insts) {
    char path[512];
    if (stream < 0) std::snprintf(path, sizeof(path), "%s_%d_inst.txt", prefix, k);
    else std::snprintf(path, sizeof(path), "%s_s%d_%d_inst.txt", prefix, stream, k);
    std::FILE* fo = std::fopen(path, "w");
    for (const auto& kv : insts)
        for (const auto& fp : kv.second.features) {
            const dynamic_vins::FeaturePoint& f = *fp.second;
            std::fprintf(fo, "%u %u %d %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.9g %d\n", kv.first, fp.first,
                         f.is_stereo ? 1 : 0, f.point[0], f.point[1], f.point[2], f.vel[0], f.vel[1], f.point_right[0],
                         f.point_right[1], f.point_right[2], f.vel_right[0], f.vel_right[1], (double)f.disp,
                         kv.second.box2d ? kv.second.box2d->track_id : -1);
        }
    std::fclose(fo);
}

// test_feature_tracker dynamic <config.yaml> <frames.bin> <n_frames> <out_prefix> <max_instances>
// FeatureTrack() of system/main.cpp:193-254 on the reference-shaped classes: reset, AddViodeInstances, TrackSemanticImage,
// InstsTrack, Output; also writes the instance table (key lost_num visible) after every frame
static int run_dynamic(int argc, char** argv) {
    if (argc < 7) { std::fprintf(stderr, "usage (dynamic)\n"); return 2; }
    const int n_frames = std::atoi(argv[4]);
    dynamic_vins::FeatureTracker::Ptr feature_tracker(new dynamic_vins::FeatureTracker(argv[2], 0, std::atoi(argv[6])));
    dynamic_vins::InstsFeatManager::Ptr insts_tracker = std::make_shared<dynamic_vins::InstsFeatManager>(std::string(argv[2]));
    const int W = feature_tracker->config().width, H = feature_tracker->config().height;
    std::ifstream fin(argv[3], std::ios::binary);
    std::vector<float> disp((size_t)W * H);
    for (size_t i = 0; i < disp.size(); i++) disp[i] = -(float)(i % 4099) - 1.f;
    for (int k = 0; k < n_frames; k++) {
        DynFrame f;
        read_dyn_frame(fin, (size_t)W * H, f);
        dynamic_vins::SemanticImage img;
        img.time0 = f.time0; img.seq = (unsigned)k;
        img.gray0 = {f.g0.data(), H, W, W};
        img.gray1 = {f.g1.data(), H, W, W};
        img.inv_merge_mask = {f.inv.data(), H, W, W};
        img.disp = {disp.data(), H, W, W * (int)sizeof(float)};
        img.exist_inst = f.exist != 0;
        img.boxes2d = f.boxes;
        dynamic_vins::FrontendFeature frame;
        frame.time = img.time0; frame.seq_id = img.seq;
        for (auto& kv : insts_tracker->instances) {                  // system/main.cpp:198-202
            kv.second.is_curr_visible = false;
            kv.second.box2d.reset();
            kv.second.box3d.reset();
        }
        insts_tracker->AddViodeInstances(img);                        // :209
        frame.features = feature_tracker->TrackSemanticImage(img);    // :250
        insts_tracker->InstsTrack(img);                               // :247
        frame.instances = insts_tracker->Output();                    // :254
        write_points(argv[5], -1, k, frame.features);
        write_instances(argv[5], -1, k, frame.instances);
        char path[512];
        std::snprintf(path, sizeof(path), "%s_%d_table.txt", argv[5], k);
        std::FILE* fo = std::fopen(path, "w");
        std::map<unsigned, const dynamic_vins::InstFeat*> sorted;
        for (auto& kv : insts_tracker->instances) sorted[kv.first] = &kv.second;
        for (auto& kv : sorted) std::fprintf(fo, "%u %d %d\n", kv.first, kv.second->lost_num, kv.second->is_curr_visible ? 1 : 0);
        std::fclose(fo);
        if (feature_tracker->prev_img.seq != (unsigned)k || feature_tracker->cur_img.gray0.data != f.g0.data()) return 4;
    }
    return 0;
}

// test_feature_tracker dynbatch <config.yaml> <frames.bin> <n_frames> <n_streams> <out_prefix> <max_instances>
// frames.bin: per frame, the n_streams stream records one after the other; BatchFeatureTracker::TrackDynamicAsync, pipelined
static int run_dynbatch(int argc, char** argv) {
    if (argc < 8) { std::fprintf(stderr, "usage (dynbatch)\n"); return 2; }
    const int n_frames = std::atoi(argv[4]), B = std::atoi(argv[5]);
    dynamic_vins::BatchFeatureTracker tracker(argv[2], B, 2, std::atoi(argv[7]));
    const int W = tracker.config().width, H = tracker.config().height;
    const size_t P = (size_t)W * H;
    std::ifstream fin(argv[3], std::ios::binary);
    std::vector<std::vector<DynFrame>> F(n_frames, std::vector<DynFrame>(B));
    std::vector<std::vector<uint8_t>> L(n_frames, std::vector<uint8_t>(B * P)), R(n_frames, std::vector<uint8_t>(B * P)),
        M(n_frames, std::vector<uint8_t>(B * P));
    for (int k = 0; k < n_frames; k++)
        for (int s = 0; s < B; s++) {
            read_dyn_frame(fin, P, F[k][s]);
            std::copy(F[k][s].g0.begin(), F[k][s].g0.end(), L[k].begin() + s * P);
            std::copy(F[k][s].g1.begin(), F[k][s].g1.end(), R[k].begin() + s * P);
            std::copy(F[k][s].inv.begin(), F[k][s].inv.end(), M[k].begin() + s * P);
        }
    auto enqueue = [&](int k) {
        std::vector<int> exist(B);
        std::vector<std::vector<dynamic_vins::Box2D::Ptr>> boxes(B);
        std::vector<double> t(B);
        for (int s = 0; s < B; s++) { exist[s] = F[k][s].exist; boxes[s] = F[k][s].boxes; t[s] = F[k][s].time0; }
        tracker.TrackDynamicAsync(L[k].data(), R[k].data(), M[k].data(), P, W, exist, boxes, t);
    };
    for (int k = 0; k < n_frames; k++) {
        enqueue(k);
        if (k > 0) {
            tracker.Wait();
            for (int s = 0; s < B; s++) { write_points(argv[6], s, k - 1, tracker.Features(s)); write_instances(argv[6], s, k - 1, tracker.InstsOutput(s)); }
        }
    }
    tracker.Wait();
    for (int s = 0; s < B; s++) { write_points(argv[6], s, n_frames - 1, tracker.Features(s)); write_instances(argv[6], s, n_frames - 1, tracker.InstsOutput(s)); }
    return 0;
}

// test_feature_tracker switch <config.yaml> <frames.bin> <calls> <out_prefix> [<back_max_level> <fb_threshold>]
// One FeatureTracker, frame k through the entry point calls[k]: 'R' TrackImage, 'S' TrackSemanticImage, 'N' TrackImageNaive.
// With the optional pair, SetLkMode sets the three sites of the CPU call pattern (both TrackImage sites and the temporal site
// of TrackSemanticImage) first.  frames.bin: per frame time0 f64, exist_inst i32, gray0, gray1, inv_merge_mask (H*W each)
static int run_switch(int argc, char** argv) {
    const std::string calls = argv[4];
    dynamic_vins::FeatureTracker tracker(argv[2]);
    if (argc >= 8)
        for (int site : {DVFE_LK_RAW_TEMPORAL, DVFE_LK_RAW_STEREO, DVFE_LK_SEMANTIC_TEMPORAL})
            tracker.SetLkMode(std::atoi(argv[6]), std::atof(argv[7]), site);
    const int W = tracker.config().width, H = tracker.config().height;
    std::ifstream fin(argv[3], std::ios::binary);
    std::vector<uint8_t> g0((size_t)W * H), g1((size_t)W * H), inv((size_t)W * H);
    for (size_t k = 0; k < calls.size(); k++) {
        dynamic_vins::SemanticImage img;
        int32_t exist = 0;
        fin.read(reinterpret_cast<char*>(&img.time0), sizeof(double));
        fin.read(reinterpret_cast<char*>(&exist), sizeof(exist));
        fin.read(reinterpret_cast<char*>(g0.data()), (std::streamsize)g0.size());
        fin.read(reinterpret_cast<char*>(g1.data()), (std::streamsize)g1.size());
        fin.read(reinterpret_cast<char*>(inv.data()), (std::streamsize)inv.size());
        img.gray0 = {g0.data(), H, W, W};
        img.gray1 = {g1.data(), H, W, W};
        img.inv_merge_mask = {inv.data(), H, W, W};
        img.exist_inst = exist != 0;
        img.seq = (unsigned)k;
        const char c = calls[k];
        const dynamic_vins::FeatureBackground fb = c == 'R' ? tracker.TrackImage(img)
                                                 : c == 'S' ? tracker.TrackSemanticImage(img)
                                                            : tracker.TrackImageNaive(img);
        write_points(argv[5], -1, (int)k, fb);
    }
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 6) { std::fprintf(stderr, "usage\n"); return 2; }
    if (std::string(argv[1]) == "switch") {
        try { return run_switch(argc, argv); } catch (const std::exception& e) { std::fprintf(stderr, "error: %s\n", e.what()); return 1; }
    }
    if (std::string(argv[1]) == "batch") {
        try { return run_batch(argc, argv); } catch (const std::exception& e) { std::fprintf(stderr, "error: %s\n", e.what()); return 1; }
    }
    if (std::string(argv[1]) == "dynamic") {
        try { return run_dynamic(argc, argv); } catch (const std::exception& e) { std::fprintf(stderr, "error: %s\n", e.what()); return 1; }
    }
    if (std::string(argv[1]) == "dynbatch") {
        try { return run_dynbatch(argc, argv); } catch (const std::exception& e) { std::fprintf(stderr, "error: %s\n", e.what()); return 1; }
    }
    try {
        dynamic_vins::FeatureTracker tracker(argv[1]);
        const int n_frames = std::atoi(argv[3]);
        const bool stereo = std::atoi(argv[4]) != 0;
        const int W = tracker.config().width, H = tracker.config().height;
        std::ifstream fin(argv[2], std::ios::binary);
        std::vector<uint8_t> g0((size_t)W * H), g1((size_t)W * H);
        for (int k = 0; k < n_frames; k++) {
            dynamic_vins::SemanticImage img;
            fin.read(reinterpret_cast<char*>(&img.time0), sizeof(double));
            fin.read(reinterpret_cast<char*>(g0.data()), (std::streamsize)g0.size());
            img.gray0 = {g0.data(), H, W, W};
            if (stereo) {
                fin.read(reinterpret_cast<char*>(g1.data()), (std::streamsize)g1.size());
                img.gray1 = {g1.data(), H, W, W};
            }
            img.seq = (unsigned)k;
            dynamic_vins::FeatureBackground fb = tracker.TrackImage(img);
            write_points(argv[5], -1, k, fb);
        }
        // the reference throws on a wrong settings path (front_end_parameters.cpp:20-22)
        bool threw = false;
        try { dynamic_vins::FeatureTracker bad("/nonexistent/config.yaml"); } catch (const std::runtime_error&) { threw = true; }
        if (!threw) { std::fprintf(stderr, "bad config path did not throw\n"); return 3; }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
