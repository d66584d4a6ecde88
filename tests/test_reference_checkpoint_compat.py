"""Checkpoint compatibility with the reference (SURVEY.md section 8 f4, README.md:154-164): the state_dict of the REAL
reference modules (the key set and shapes of the official pose_hrnet_* / pose_resnet_* checkpoints, which are plain
state_dicts of these modules) is accepted by the plan's strict packer, in both checkpoint formats the reference loads
(SimpleHRNet.py:117-121), and every tensor lands where the plan says.  The reference modules' keys, shapes and dtypes
are stored in tests/golden/reference_state_dicts.npz (make_golden.py); the values are seeded random.  CPU only."""
import os

import numpy as np
import pytest
import torch

from simple_hrnet_b200.engine import Plan, expected_state_dict_keys, pack_state_dict


def _reference_state_dict(golden_dir, tag):
    """A state_dict with the reference module's keys, order, shapes and dtypes; values seeded random (positive, so that
    running_var is a valid variance)."""
    g = np.load(os.path.join(golden_dir, "reference_state_dicts.npz"))
    dims, pos, sd = g[tag + "_dims"], 0, {}
    gen = torch.Generator().manual_seed(0)
    for key, ndim, dtype in zip(g[tag + "_keys"], g[tag + "_ndim"], g[tag + "_dtypes"]):
        shape = tuple(int(d) for d in dims[pos:pos + ndim])
        pos += ndim
        dtype = getattr(torch, str(dtype))
        sd[str(key)] = (torch.rand(shape, generator=gen) + 0.5).to(dtype) if dtype.is_floating_point else torch.zeros(shape, dtype=dtype)
    assert pos == len(dims)
    return sd


@pytest.mark.parametrize("arch,c,res", [("hrnet", 32, (256, 192)), ("hrnet", 48, (384, 288)), ("poseresnet", 50, (256, 192)),
                                         ("poseresnet", 101, (256, 192))])
def test_real_module_state_dict_is_accepted(golden_dir, arch, c, res):
    sd = _reference_state_dict(golden_dir, f"{arch}{c}")
    plan = Plan(arch, c, 17, res, 2)
    req, opt = expected_state_dict_keys(plan.infos)
    assert set(req) | opt == set(sd.keys())                       # exactly the reference's key set (1,754 keys for HRNet)
    buf = pack_state_dict(sd, plan.infos, plan.weight_bytes)
    buf2 = pack_state_dict({"model": sd, "epoch": 3}, plan.infos, plan.weight_bytes)   # training checkpoints (SimpleHRNet.py:118-119)
    assert np.array_equal(buf, buf2)
    # spot-check the layout: first conv (fp32 [cout][kh][kw][cin]) and the head bias
    pi = plan.infos[0]
    w = sd[pi.conv_key.decode() + ".weight"].permute(0, 2, 3, 1).contiguous().numpy().astype(np.float32 if pi.w_f32 else np.float16)
    assert np.array_equal(np.frombuffer(buf[pi.w_offset:pi.w_offset + w.nbytes].tobytes(), dtype=w.dtype), w.ravel())
    head = [p for p in plan.infos if p.conv_key.decode() == "final_layer"][0]
    b = sd["final_layer.bias"].numpy()
    assert np.array_equal(np.frombuffer(buf[head.bias_offset:head.bias_offset + b.nbytes].tobytes(), dtype=np.float32), b)
    # a checkpoint with a missing / an unexpected key is rejected like load_state_dict(strict=True)
    bad = dict(sd); bad.pop("final_layer.bias")
    with pytest.raises(RuntimeError, match="Missing key"):
        pack_state_dict(bad, plan.infos, plan.weight_bytes)
    bad = dict(sd); bad["module.conv1.weight"] = sd["conv1.weight"]
    with pytest.raises(RuntimeError, match="Unexpected key"):
        pack_state_dict(bad, plan.infos, plan.weight_bytes)
