// dvfe_config_from_yaml — replaces fe_para::SetParameters (dynamic_vins/src/front_end/front_end_parameters.cpp:17-40),
// the cfg keys the path reads (dynamic_vins/src/utils/parameters.cpp:19-147: num_of_cam, image_width/height,
// cam0_calib, cam1_calib) and the camodocal PINHOLE yaml reader
// (/root/reference/camera_models/src/camera_models/PinholeCamera.cc:80-140, readFromYamlFile), which dvfe_camera_from_yaml
// exposes on its own for per-stream calibrations.
// The reference parses with cv::FileStorage; the files are flat "key: value" yaml (OpenCV "%YAML:1.0" dialect)
// with at most one level of nesting and unique leaf names, which is all this reader supports.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>

#include "../../include/dvfe.h"
#include "../../include/dvfe/reject_with_f.h"

void dvfe_set_error(const char* fmt, ...);

namespace {
std::string trim(const std::string& s) {
    size_t b = s.find_first_not_of(" \t\r\n\"");
    if (b == std::string::npos) return "";
    size_t e = s.find_last_not_of(" \t\r\n\"");
    return s.substr(b, e - b + 1);
}

bool read_flat_yaml(const std::string& path, std::map<std::string, std::string>& kv) {
    FILE* f = fopen(path.c_str(), "r");
    if (!f) return false;
    char line[4096];
    while (fgets(line, sizeof(line), f)) {
        std::string s(line);
        const size_t hash = s.find('#');
        if (hash != std::string::npos) s = s.substr(0, hash);
        if (s.empty() || s[0] == '%' || s.compare(0, 3, "---") == 0) continue;
        const size_t colon = s.find(':');
        if (colon == std::string::npos) continue;
        const std::string key = trim(s.substr(0, colon));
        const std::string val = trim(s.substr(colon + 1));
        if (!key.empty() && !val.empty() && kv.find(key) == kv.end()) kv[key] = val;
    }
    fclose(f);
    return true;
}

bool get_int(const std::map<std::string, std::string>& kv, const char* key, int* out) {
    auto it = kv.find(key);
    if (it == kv.end()) return false;
    *out = (int)strtod(it->second.c_str(), nullptr);
    return true;
}
bool get_double(const std::map<std::string, std::string>& kv, const char* key, double* out) {
    auto it = kv.find(key);
    if (it == kv.end()) return false;
    *out = strtod(it->second.c_str(), nullptr);
    return true;
}

int read_camera(const std::string& path, dvfe_camera* cam) {
    std::map<std::string, std::string> kv;
    if (!read_flat_yaml(path, kv)) {
        dvfe_set_error("ERROR: Wrong path to camera calibration:%s", path.c_str());
        return DVFE_ERR_CONFIG;
    }
    auto mt = kv.find("model_type");
    if (mt == kv.end() || mt->second != "PINHOLE") {
        dvfe_set_error("camera %s: only model_type PINHOLE is supported on this path", path.c_str());
        return DVFE_ERR_CONFIG;
    }
    memset(cam, 0, sizeof(*cam));
    if (!get_double(kv, "fx", &cam->fx) || !get_double(kv, "fy", &cam->fy) || !get_double(kv, "cx", &cam->cx) ||
        !get_double(kv, "cy", &cam->cy)) {
        dvfe_set_error("camera %s: projection_parameters missing", path.c_str());
        return DVFE_ERR_CONFIG;
    }
    get_double(kv, "k1", &cam->k1); get_double(kv, "k2", &cam->k2);
    get_double(kv, "p1", &cam->p1); get_double(kv, "p2", &cam->p2);
    return DVFE_OK;
}
}  // namespace

extern "C" int dvfe_camera_from_yaml(const char* path, dvfe_camera* cam) {
    if (!path || !cam) { dvfe_set_error("camera_from_yaml: null argument"); return DVFE_ERR_INVALID; }
    dvfe_camera c;
    const int rc = read_camera(path, &c);
    if (rc == DVFE_OK) *cam = c;
    return rc;
}

extern "C" int dvfe_f_threshold_from_yaml(const char* path, double* f) {
    if (!path || !f) { dvfe_set_error("f_threshold_from_yaml: null argument"); return DVFE_ERR_INVALID; }
    std::map<std::string, std::string> kv;
    if (!read_flat_yaml(path, kv)) {
        dvfe_set_error("ERROR: Wrong path to settings:%s", path);
        return DVFE_ERR_CONFIG;
    }
    double v = 0.0;                           // fs["F_threshold"] >> F_threshold: 0 when the key is absent
    get_double(kv, "F_threshold", &v);
    *f = v;
    return DVFE_OK;
}

extern "C" int dvfe_config_from_yaml(const char* config_path, dvfe_config* cfg) {
    if (!config_path || !cfg) { dvfe_set_error("config_from_yaml: null argument"); return DVFE_ERR_INVALID; }
    std::map<std::string, std::string> kv;
    if (!read_flat_yaml(config_path, kv)) {
        dvfe_set_error("ERROR: Wrong path to settings:%s", config_path);      // front_end_parameters.cpp:20-22
        return DVFE_ERR_CONFIG;
    }
    memset(cfg, 0, sizeof(*cfg));
    cfg->n_streams = 1;
    cfg->lk_max_level = 3;
    cfg->max_instances = 0;
    cfg->flow_back = 1;
    cfg->mask_morphology_size = 5;
    if (!get_int(kv, "max_cnt", &cfg->max_cnt) || !get_int(kv, "min_dist", &cfg->min_dist) ||
        !get_int(kv, "image_width", &cfg->width) || !get_int(kv, "image_height", &cfg->height)) {
        dvfe_set_error("settings %s: max_cnt / min_dist / image_width / image_height missing", config_path);
        return DVFE_ERR_CONFIG;
    }
    get_int(kv, "max_dynamic_cnt", &cfg->max_dynamic_cnt);
    get_int(kv, "min_dynamic_dist", &cfg->min_dynamic_dist);
    get_int(kv, "flow_back", &cfg->flow_back);
    get_int(kv, "use_mask_morphology", &cfg->use_mask_morphology);
    get_int(kv, "mask_morphology_size", &cfg->mask_morphology_size);
    int num_of_cam = 1;
    get_int(kv, "num_of_cam", &num_of_cam);
    cfg->stereo = num_of_cam == 2;
    auto st = kv.find("slam_type");
    if (st != kv.end() && st->second == "dynamic") cfg->max_instances = 32;
    std::string dir(config_path);
    const size_t slash = dir.find_last_of('/');
    dir = slash == std::string::npos ? std::string("") : dir.substr(0, slash + 1);
    auto c0 = kv.find("cam0_calib");
    if (c0 == kv.end()) { dvfe_set_error("settings %s: cam0_calib missing", config_path); return DVFE_ERR_CONFIG; }
    int rc = read_camera(dir + c0->second, &cfg->cam0);
    if (rc != DVFE_OK) return rc;
    cfg->cam1 = cfg->cam0;
    auto c1 = kv.find("cam1_calib");
    if (cfg->stereo && c1 != kv.end()) {
        rc = read_camera(dir + c1->second, &cfg->cam1);
        if (rc != DVFE_OK) return rc;
    }
    return DVFE_OK;
}
