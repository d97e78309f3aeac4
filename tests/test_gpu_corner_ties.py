"""Corner selection under heavy ties and past the capacity of its candidate buffer.

Natural and random images almost never give two equal strongest responses, so the (response desc, address desc) order that
cv::goodFeaturesToTrack applies (std::sort with greaterThanPtr) is not exercised by the other tests through the radix select,
the per-cell sort and the bitonic merge of the kernels.  Here:
  * a periodic plateau image I(x, y) = f[x % 3] + f[y % 3] whose response map is constant over the interior (thousands of
    exactly equal local maxima), through the fused op and through `eig=` cv2's own map;
  * response maps with 2-4 distinct levels, against a brute-force restatement of cv2's rule written here, independent of
    oracle/spec.c;
  * more local maxima than the candidate buffer holds (W*H/4 + 4096): the op fails with DVFE_ERR_CAPACITY, and in a
    pipelined tracker only the wait for the step that overflowed reports it while the other stream stays exact."""
import cv2
import numpy as np
import pytest

import dynamic_vins_b200 as dv
from dynamic_vins_b200 import BatchTracker, make_config, ops, synth
from oracle import cv_front_end as cvfe
from oracle import spec

pytestmark = pytest.mark.gpu


def plateau(h, w, f=(0, 40, 110)):
    f = np.asarray(f, np.int32)
    yy, xx = np.mgrid[0:h, 0:w]
    return (f[xx % 3] + f[yy % 3]).astype(np.uint8)


def holey_mask(h, w, seed=3):
    rng = np.random.default_rng(seed)
    m = np.full((h, w), 255, np.uint8)
    for _ in range(12):
        y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
        m[max(0, y - 4):y + 5, max(0, x - 6):x + 7] = 0
    m[:, w // 2] = 0
    return m


def brute_gftt(eig, mask, K, md, unmasked_max=False):
    """cv::goodFeaturesToTrack's selection on a response map, restated directly: maximum over the mask (or the whole map),
    strict threshold against (float)(max * 0.01), 3x3 local maxima of the thresholded map, 1 <= x < W-1, 1 <= y < H-1,
    order (value desc, address desc), greedy acceptance while the squared distance to every accepted corner is >= md^2"""
    eig = np.asarray(eig, np.float32)
    h, w = eig.shape
    sel = mask != 0 if (mask is not None and not unmasked_max) else np.ones(eig.shape, bool)
    thr = np.float32(float(eig[sel].max()) * 0.01)
    t = np.where(eig > thr, eig, np.float32(0))
    pad = np.pad(t, 1, constant_values=-np.inf)
    dil = np.max([pad[dy:dy + h, dx:dx + w] for dy in range(3) for dx in range(3)], axis=0)
    cand = [(float(t[y, x]), y * w + x) for y in range(1, h - 1) for x in range(1, w - 1)
            if t[y, x] != 0 and t[y, x] == dil[y, x] and (mask is None or mask[y, x] != 0)]
    cand.sort(key=lambda c: (-c[0], -c[1]))
    out = []
    for _, a in cand:
        y, x = divmod(a, w)
        if all((x - px) ** 2 + (y - py) ** 2 >= md * md for px, py in out):
            out.append((x, y))
            if len(out) == K:
                break
    return np.asarray(out, np.float32).reshape(-1, 2)


@pytest.mark.parametrize("cuda_rule", [False, True])
@pytest.mark.parametrize("masked", [False, True])
def test_plateau_ties(masked, cuda_rule):
    img = plateau(72, 72)
    eig_spec = spec.min_eigen_val(img)
    assert np.unique(eig_spec[2:-2, 2:-2]).size == 1               # one value over the whole interior
    mask = holey_mask(72, 72) if masked else None
    eig_cv = cv2.cornerMinEigenVal(img, 3, ksize=3)
    for K in (1, 50, 2048):                                       # 2048: the op's largest max_corners
        for md in (1, 1.5, 2, 5, 7):
            got = ops.good_features(img, K, 0.01, md, mask=mask, cuda_semantics=cuda_rule)
            want = spec.gftt_select(eig_spec, mask, K, 0.01, md, unmasked_max=cuda_rule)[0]
            assert got.tobytes() == want.tobytes(), (K, md)
            assert len(got) == min(K, len(want)) and len(got) >= 1
            if not cuda_rule:
                p = cv2.goodFeaturesToTrack(img, K, 0.01, md, mask=mask)
                p = np.zeros((0, 2), np.float32) if p is None else p.reshape(-1, 2)
                assert ops.good_features(None, K, 0.01, md, mask=mask, eig=eig_cv).tobytes() == p.tobytes(), (K, md)
            if md == 1 and K == 2048:
                assert len(got) > 1000


@pytest.mark.parametrize("shape", [(61, 77), (128, 128), (33, 200)])
def test_quantised_maps_vs_brute_force(shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    h, w = shape
    for trial in range(6):
        n_levels = 2 + trial % 3
        levels = np.sort(rng.choice([0.0, 1e-4, 2.5e-3, 0.37, 1.0, 3.5], n_levels, replace=False)).astype(np.float32)
        eig = levels[rng.integers(0, n_levels, (h, w))]
        mask = holey_mask(h, w, trial) if trial % 2 else None
        for K, md in ((1, 1), (40, 1.5), (300, 2), (2048, 1), (20, 5)):
            for rule in (False, True):
                got = ops.good_features(None, K, 0.01, md, mask=mask, eig=eig, cuda_semantics=rule)
                want = brute_gftt(eig, mask, K, md, unmasked_max=rule)
                assert got.tobytes() == want.tobytes(), (trial, K, md, rule)


def test_candidate_buffer_overflow_op():
    h, w = 200, 240
    img = plateau(h, w)
    with pytest.raises(dv.DvfeError) as e:
        ops.good_features(img, 500, 0.01, 5)
    assert e.value.code == -4
    assert len(ops.good_features(plateau(72, 72), 500, 0.01, 5)) > 0     # the op works again afterwards


def test_candidate_buffer_overflow_in_one_stream_one_step():
    """B = 2 tracker of the C5 shape, pipelined: stream 1 gets a plateau left image at step 2 (~ 900 000 local maxima > the
    W*H/4 + 4096 the buffer holds).  Only the wait for step 2 raises DVFE_ERR_CAPACITY; stream 0 is exact on every frame."""
    name, B, T = "c5_zed_streams", 2, 6
    c = dict(synth.CONFIGS[name]); c.pop("n_objects"); c.pop("config_id")
    trk = BatchTracker(make_config(n_streams=B, **c))
    sts = [synth.make_stream(name, 90 + s) for s in range(B)]
    frames = [[st.frame(k) for k in range(T)] for st in sts]
    frames[1][2].gray0 = plateau(c["height"], c["width"])
    P = cvfe.FrontEndParams(max_cnt=c["max_cnt"], min_dist=c["min_dist"], is_stereo=True, arith="exact")
    fe = cvfe.FrontEnd(P, c["cam0"], c["cam1"], "raw")
    want = [fe.step(fr)["features"] for fr in frames[0]]
    from test_gpu_exact_frame_step import assert_records
    raised = []
    for k in range(T + 1):
        if k < T:
            trk.track_image_async(np.stack([frames[s][k].gray0 for s in range(B)]),
                                  np.stack([frames[s][k].gray1 for s in range(B)]), frames[0][k].time0)
        if k > 0:
            try:
                trk.wait()
            except dv.DvfeError as e:
                assert e.code == -4
                raised.append(k - 1)
            assert_records(trk.features(0), want[k - 1], f"stream 0 frame {k - 1}")
    assert raised == [2]
    trk.close()
