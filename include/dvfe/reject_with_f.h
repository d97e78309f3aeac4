/* dvfe/reject_with_f.h -- companion of dvfe.h: epipolar outlier rejection inside the frame step.  The functions are part of
 * libdvfe (same library, same error codes, same dvfe_tracker handle); include this header after or instead of dvfe.h. */
#ifndef DVFE_REJECT_WITH_F_H_
#define DVFE_REJECT_WITH_F_H_
#include "../dvfe.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Epipolar outlier rejection inside the frame step: VINS-Mono's rejectWithF (FeatureTracker::RejectWithF,
 * front_end/background_tracker.cpp:520-550, whose call the reference leaves commented out), for every stream of every
 * background step (TrackImage, TrackSemanticImage, TrackImageNaive and the background half of dynamic mode, through every entry
 * point).  Tracker-wide and off by default; f_threshold = fe_para::F_threshold (dvfe_f_threshold_from_yaml).
 *   0     off (default): every step is exactly the step without this call (same graphs, same kernel launches)
 *   > 0   on from the next submitted step: for each stream that ran the temporal LK, after the LK survivors are known and before
 *         the disc mask and the detection, n = the number of survivors (current point, previous point, in id order).  With
 *         n >= 8 both lists are lifted with the stream's cam0 (dvfe_set_stream_camera), re-projected with 460 about
 *         (width/2, height/2) and given to cv::findFundamentalMat(cur, prev, FM_RANSAC, f_threshold, 0.99) with a fresh
 *         cv::RNG(-1) per stream and step (LMedS for 8 <= n < 15, as in OpenCV) -- the computation of dvfe_op_reject_with_f.
 *         Points with status 0 are removed as ReduceVector removes them (ids, track_cnt, positions, velocity maps), so the
 *         detection of the same step may fill their area and slots; stereo LK, lifting and velocities run on what is left.
 *         When no model is found (every 7-point sample degenerate, e.g. all survivors at one position) every point is kept.  This
 *         differs on purpose from dvfe_op_reject_with_f, which reports all zeros then: OpenCV returns an empty mask, which
 *         VINS-Mono's reduceVector would read past.  Adds one kernel launch per step (and stream group) with a temporal LK.
 * Skipped streams, first frames and DVFE_FRAME_RESET streams (no temporal LK) are unchanged, and so are instances
 * (InstsFeatManager::RejectWithF stays the seam op).  Negative or non-finite f_threshold: DVFE_ERR_INVALID, nothing changed.
 * With stream groups the setting goes to every group. */
int dvfe_set_reject_with_f(dvfe_tracker* t, double f_threshold);

/* fe_para::F_threshold of a front-end settings file (front_end/front_end_parameters.cpp), read like dvfe_config_from_yaml reads
 * the other keys: *f = the value, 0 when the key is absent (cv::FileStorage reads a missing key as 0).  DVFE_ERR_CONFIG for a
 * bad path.  Needs no device. */
int dvfe_f_threshold_from_yaml(const char* path, double* f);

#ifdef __cplusplus
}
#endif
#endif /* DVFE_REJECT_WITH_F_H_ */
