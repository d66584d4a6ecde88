"""
Generates the committed golden fixtures in tests/golden/ by running the REAL
reference (stefanopini/simple-HRNet, read-only at /root/reference) on CPU in the
build container.  The reference ships no tests or golden vectors for this path
(SURVEY.md section 4), so these fixtures are what pins the oracle (oracle/hrnet_oracle.py)
and, through it, the CUDA path.

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz

Each fixture records the seeds needed to regenerate weights and inputs through
oracle.make_state_dict / the generators below (weights are 114-254 MB and are never
committed), plus the outputs of the reference classes:

  * models_.hrnet.HRNet / models_.poseresnet.PoseResNet  .forward      (model boundary)
  * SimpleHRNet.SimpleHRNet(...).predict                               (API boundary)

It also asserts, while generating, that the oracle restatement is bit-identical to the
reference on every fixture (so a drift in either is caught here first).
"""
import hashlib
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("SIMPLE_HRNET_REF", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

from oracle import hrnet_oracle as O  # noqa: E402


def model_input(n, h, w, seed):
    return torch.randn(n, 3, h, w, generator=torch.Generator().manual_seed(seed))


def crop_u8(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


def gaps(hm):
    flat = torch.from_numpy(hm).reshape(hm.shape[0], hm.shape[1], -1)
    t = flat.topk(2, dim=2).values
    return (t[..., 0] - t[..., 1]).numpy()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def build_ref_model(arch, c, sd):
    from models_.hrnet import HRNet
    from models_.poseresnet import PoseResNet
    m = HRNet(c, 17) if arch == "hrnet" else PoseResNet(c, 17)
    m.load_state_dict(sd, strict=True)
    return m.eval()


def model_fixture(name, arch, c, n, h, w, wseed, bn, xseed, store_heatmaps=True):
    spec = O.hrnet_param_spec(c, 17) if arch == "hrnet" else O.poseresnet_param_spec(c, 17)
    sd = O.make_state_dict(spec, seed=wseed, bn=bn)
    x = model_input(n, h, w, xseed)
    with torch.no_grad():
        hm = build_ref_model(arch, c, sd)(x).numpy()
    ohm = (O.hrnet_forward(sd, x) if arch == "hrnet" else O.poseresnet_forward(sd, x, c)).numpy()
    assert np.array_equal(hm, ohm), f"{name}: oracle != reference"
    boxes = np.repeat(np.asarray([[0, 0, w, h]], dtype=np.float32), n, axis=0)
    pts, idx = O.decode_joints(hm, boxes)
    out = dict(arch=arch, c=c, n=n, h=h, w=w, wseed=wseed, bn=bn, xseed=xseed,
               argmax=idx, pts=pts, gaps=gaps(hm), hm_sha256=sha(hm),
               hm_stats=np.asarray([hm.min(), hm.mean(), hm.max()], dtype=np.float64))
    if store_heatmaps:
        out["heatmaps"] = hm
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print(f"{name}: hm [{hm.min():.4f},{hm.max():.4f}] min gap {out['gaps'].min():.3e} sha {out['hm_sha256'][:12]}")


def predict_fixture(name, c, res, img_shape, wseed, bn, iseed):
    """API boundary: the reference's SimpleHRNet.predict on uint8 BGR crops."""
    from SimpleHRNet import SimpleHRNet
    spec = O.hrnet_param_spec(c, 17)
    sd = O.make_state_dict(spec, seed=wseed, bn=bn)
    img = crop_u8(img_shape, iseed)
    with tempfile.TemporaryDirectory() as td:
        ck = os.path.join(td, "w.pth")
        torch.save(sd, ck)
        m = SimpleHRNet(c, 17, ck, resolution=res, multiperson=False, return_heatmaps=True,
                        return_bounding_boxes=True, max_batch_size=64, device=torch.device("cpu"))
        hm, boxes, pts = m.predict(img)
    ohm, oboxes, opts = O.predict(sd, img, res)
    assert np.array_equal(hm, ohm) and np.array_equal(boxes, oboxes) and np.array_equal(pts, opts), \
        f"{name}: oracle predict != reference predict"
    np.savez_compressed(os.path.join(HERE, name + ".npz"), c=c, res=np.asarray(res), img_shape=np.asarray(img_shape),
                        wseed=wseed, bn=bn, iseed=iseed, heatmaps=hm, boxes=boxes, pts=pts, gaps=gaps(hm),
                        hm_sha256=sha(hm))
    print(f"{name}: pts shape {pts.shape} boxes {boxes[0]} hm [{hm.min():.4f},{hm.max():.4f}]")


def decode_fixture():
    """Argmax-decode boundary incl. exact ties and non-trivial boxes: run the reference's own
    decode loop (SimpleHRNet.py:296-308) by monkey-patching `self.model` with a lookup."""
    rng = np.random.default_rng(7)
    n, J, Hh, Wh = 6, 17, 16, 12
    hm = rng.standard_normal((n, J, Hh, Wh)).astype(np.float32)
    hm[0, 0] = 0.25                      # all-equal map: first index must win
    hm[1, 3, 5, 7] = hm[1, 3, 9, 2] = 9.0  # exact tie: lower flat index wins
    hm[2, 4, Hh - 1, Wh - 1] = 50.0      # last element
    hm[3, 5] = -np.abs(hm[3, 5]) - 1      # all negative
    from SimpleHRNet import SimpleHRNet

    class _Stub:
        def __call__(self, images):
            return torch.from_numpy(hm[: images.shape[0]])

    m = SimpleHRNet.__new__(SimpleHRNet)
    m.resolution = (Hh * 4, Wh * 4); m.nof_joints = J; m.multiperson = False
    m.return_heatmaps = False; m.return_bounding_boxes = True; m.max_batch_size = 64
    m.device = torch.device("cpu"); m.model = _Stub(); m.interpolation = 2
    from torchvision.transforms import transforms
    m.transform = transforms.Compose([transforms.ToTensor(),
                                      transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    imgs = crop_u8((n, 123, 77, 3), 11)   # odd original size -> non-trivial float box scaling
    boxes, pts = m.predict(imgs)
    opts, oidx = O.decode_joints(hm, boxes)
    assert np.array_equal(pts[:, 0], opts), "decode oracle != reference"
    np.savez_compressed(os.path.join(HERE, "decode_edge.npz"), heatmaps=hm, boxes=boxes, pts=opts, argmax=oidx)
    print("decode_edge: ok", boxes[0])


STATE_DICT_CONFIGS = [("hrnet", 32), ("hrnet", 48), ("poseresnet", 50), ("poseresnet", 101)]


def state_dict_fixture():
    """Key set, shapes and dtypes of the reference modules' state_dicts (the layout of the official pose_hrnet_* /
    pose_resnet_* checkpoints), in the modules' own order."""
    from models_.hrnet import HRNet
    from models_.poseresnet import PoseResNet
    out = {}
    for arch, c in STATE_DICT_CONFIGS:
        sd = (HRNet(c, 17) if arch == "hrnet" else PoseResNet(c, 17)).state_dict()
        tag = f"{arch}{c}"
        out[tag + "_keys"] = np.asarray(list(sd.keys()))
        out[tag + "_ndim"] = np.asarray([t.dim() for t in sd.values()], dtype=np.int32)
        out[tag + "_dims"] = np.asarray([d for t in sd.values() for d in t.shape], dtype=np.int32)
        out[tag + "_dtypes"] = np.asarray([str(t.dtype).replace("torch.", "") for t in sd.values()])
        print(f"reference_state_dicts: {tag} {len(sd)} keys")
    np.savez_compressed(os.path.join(HERE, "reference_state_dicts.npz"), **out)


SEAM_CASES = [("hrnet", 32, (256, 192), 6), ("hrnet", 48, (384, 288), 5), ("poseresnet", 50, (256, 192), 3)]
SEAM_SAMPLE = 2048


def seam_fixture():
    """The reference's SimpleHRNet(device=cpu, max_batch_size=4).predict on one image at another resolution (it is resized)
    and on a stack longer than max_batch_size (it is chunked).  Heat-maps are too large to store whole: a fixed sample of
    SEAM_SAMPLE values per input, max |heat-map| and the top-1 / top-2 gaps are kept, boxes and joints in full."""
    from SimpleHRNet import SimpleHRNet
    out = {}
    for arch, c, res, batch in SEAM_CASES:
        spec = O.hrnet_param_spec(c, 17) if arch == "hrnet" else O.poseresnet_param_spec(c, 17)
        sd = O.make_state_dict(spec, seed=0, bn="default")
        with tempfile.TemporaryDirectory() as td:
            ck = os.path.join(td, "w.pth")
            torch.save(sd, ck)
            m = SimpleHRNet(c, 17, ck, model_name="HRNet" if arch == "hrnet" else "PoseResNet", resolution=res,
                            multiperson=False, return_heatmaps=True, return_bounding_boxes=True, max_batch_size=4,
                            device=torch.device("cpu"))
        rng = np.random.default_rng(7)
        img = rng.integers(0, 256, (300, 210, 3), dtype=np.uint8)
        stack = rng.integers(0, 256, (batch, res[0], res[1], 3), dtype=np.uint8)
        for kind, inp in (("img", img), ("stack", stack)):
            hm, boxes, pts = m.predict(inp)
            ohm, oboxes, opts = O.predict(sd, inp, res, model=arch, resnet_size=c)
            assert np.array_equal(hm, ohm) and np.array_equal(boxes, oboxes) and np.array_equal(pts, opts), \
                f"{arch}{c} {kind}: oracle predict != reference predict"
            tag = f"{arch}{c}_{kind}"
            at = np.sort(np.random.default_rng(0).choice(hm.size, SEAM_SAMPLE, replace=False)).astype(np.int64)
            out.update({tag + "_hm_shape": np.asarray(hm.shape), tag + "_hm_at": at, tag + "_hm_values": hm.ravel()[at],
                        tag + "_hm_absmax": np.float32(np.abs(hm).max()), tag + "_gaps": gaps(hm),
                        tag + "_boxes": boxes, tag + "_pts": pts})
            print(f"reference_seam_predict: {tag} hm {hm.shape} max|hm| {np.abs(hm).max():.4f} pts {pts.shape}")
    np.savez_compressed(os.path.join(HERE, "reference_seam_predict.npz"), **out)


if __name__ == "__main__":
    torch.set_num_threads(8)             # tests/test_oracle.py replays the fixtures bit for bit with the same count
    state_dict_fixture()
    seam_fixture()
    decode_fixture()
    # tiny net-level fixture for fast CPU tests (resolution must be a multiple of 32)
    model_fixture("w32_64x64_n2_rand", "hrnet", 32, 2, 64, 64, wseed=3, bn="random", xseed=5)
    # BASELINE config 1 (API boundary) and config 2/3 shapes at the model boundary
    predict_fixture("w32_256x192_predict", 32, (256, 192), (256, 192, 3), wseed=0, bn="default", iseed=0)
    model_fixture("w32_256x192_n2_default", "hrnet", 32, 2, 256, 192, wseed=0, bn="default", xseed=0)
    model_fixture("w32_256x192_n2_rand", "hrnet", 32, 2, 256, 192, wseed=1, bn="random", xseed=1)
    model_fixture("w48_384x288_n1_default", "hrnet", 48, 1, 384, 288, wseed=0, bn="default", xseed=0)
    model_fixture("w48_384x288_n4_default_summary", "hrnet", 48, 4, 384, 288, wseed=0, bn="default", xseed=2,
                  store_heatmaps=False)
    model_fixture("poseresnet50_256x192_n1_default", "poseresnet", 50, 1, 256, 192, wseed=0, bn="default", xseed=0)
