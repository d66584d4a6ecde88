"""CPU tests: the oracle restatement replayed against the fixtures generated from the real
reference (tests/golden/make_golden.py).  Bit-exact: same aten/numpy ops, same inputs, same CPU thread count."""
import os

import numpy as np
import pytest
import torch

from oracle import hrnet_oracle as O

# make_golden.py runs the reference with this many CPU threads.  oneDNN splits the reductions of an fp32 convolution by
# thread count, so a replay with another count differs in the last bits (measured: up to 7e-8 on the PoseResNet-50 maps).
GOLDEN_THREADS = 8


@pytest.fixture(autouse=True, scope="module")
def _golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False)


def _x(g):
    return torch.randn(int(g["n"]), 3, int(g["h"]), int(g["w"]), generator=torch.Generator().manual_seed(int(g["xseed"])))


@pytest.mark.parametrize("name", ["w32_64x64_n2_rand", "w32_256x192_n2_default", "w32_256x192_n2_rand"])
def test_hrnet_forward_matches_reference_fixture(golden_dir, name):
    g = _load(golden_dir, name)
    sd = O.make_state_dict(O.hrnet_param_spec(int(g["c"]), 17), seed=int(g["wseed"]), bn=str(g["bn"]))
    hm = O.hrnet_forward(sd, _x(g)).numpy()
    assert np.array_equal(hm, g["heatmaps"])
    boxes = np.repeat(np.asarray([[0, 0, int(g["w"]), int(g["h"])]], dtype=np.float32), int(g["n"]), axis=0)
    pts, idx = O.decode_joints(hm, boxes)
    assert np.array_equal(idx, g["argmax"]) and np.array_equal(pts, g["pts"])


def test_w48_forward_matches_reference_fixture(golden_dir):
    g = _load(golden_dir, "w48_384x288_n1_default")
    sd = O.make_state_dict(O.hrnet_param_spec(48, 17), seed=int(g["wseed"]), bn=str(g["bn"]))
    hm = O.hrnet_forward(sd, _x(g)).numpy()
    assert np.array_equal(hm, g["heatmaps"])


def test_poseresnet_forward_matches_reference_fixture(golden_dir):
    g = _load(golden_dir, "poseresnet50_256x192_n1_default")
    sd = O.make_state_dict(O.poseresnet_param_spec(50, 17), seed=int(g["wseed"]), bn=str(g["bn"]))
    hm = O.poseresnet_forward(sd, _x(g), 50).numpy()
    assert np.array_equal(hm, g["heatmaps"])


def test_predict_matches_reference_fixture(golden_dir):
    """BASELINE config 1: SimpleHRNet.predict on one uint8 crop, multiperson=False."""
    g = _load(golden_dir, "w32_256x192_predict")
    sd = O.make_state_dict(O.hrnet_param_spec(32, 17), seed=int(g["wseed"]), bn=str(g["bn"]))
    img = np.random.default_rng(int(g["iseed"])).integers(0, 256, tuple(g["img_shape"]), dtype=np.uint8)
    hm, boxes, pts = O.predict(sd, img, tuple(int(v) for v in g["res"]))
    assert np.array_equal(hm, g["heatmaps"]) and np.array_equal(boxes, g["boxes"]) and np.array_equal(pts, g["pts"])
    assert pts.shape == (1, 17, 3)
    # (y, x, conf): y first (SimpleHRNet.py:198,306-308); boxes = [0,0,W,H] so y = 4*row, x = 4*col
    idx = np.argmax(hm.reshape(1, 17, -1), axis=2)
    assert np.array_equal(pts[0, :, 0], 4.0 * (idx[0] // 48)) and np.array_equal(pts[0, :, 1], 4.0 * (idx[0] % 48))


def test_decode_edge_cases(golden_dir):
    """Ties (first occurrence), all-equal maps, negative maps, last element, non-integer box scale."""
    g = _load(golden_dir, "decode_edge")
    pts, idx = O.decode_joints(g["heatmaps"], g["boxes"])
    assert np.array_equal(pts, g["pts"]) and np.array_equal(idx, g["argmax"])
    assert idx[0, 0] == 0                       # all-equal map -> index 0
    assert idx[1, 3] == 5 * 12 + 7              # tie -> lower flat index
    assert idx[2, 4] == 16 * 12 - 1             # last element
    assert pts[3, 5, 2] < 0                     # confidence is the raw (negative) heatmap value


def test_decode_empty_batch():
    pts, idx = O.decode_joints(np.zeros((0, 17, 8, 6), np.float32), np.zeros((0, 4), np.float32))
    assert pts.shape == (0, 17, 3) and idx.shape == (0, 17)


def test_predict_wrong_format():
    with pytest.raises(ValueError, match="Wrong image format"):
        O.predict({}, np.zeros((4, 4), np.uint8), (64, 64))
