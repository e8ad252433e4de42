"""The two fixed-window paths, composed from oracle.ref_preprocess's resize and enhance_thermal_fixed_range, against the
live reference's recorded outputs (tests/golden/preprocess_kat.npz, key <tag>_fixed: [0] the inference path, [1] the
train path; oracle/gen_golden.py).  The GPU tests use these compositions as their oracle."""
import hashlib
import os

import numpy as np
import pytest

from oracle import ref_preprocess

SIZES = ((224, 224), (512, 384), (333, 217))      # (w, h), cv2 order


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def train_path_fixed_range(raw_u16, dst_hw):
    """data/dataset_loader.py:237-249 with the fixed window at :111 : u16 -> resize (u16) -> f32 raw counts -> 3ch
    -> enhance_thermal_fixed_range(normalized=False) (the values are raw counts).  Returns out[3,h,w]."""
    r = ref_preprocess.resize_bilinear(raw_u16, dst_hw)
    return ref_preprocess.enhance_thermal_fixed_range(np.repeat(r.astype(np.float32)[None], 3, 0), normalized=False)


def inference_path_fixed_range(raw_u16, dst_hw):
    """thermal_dustr_inference.py:25-60 with the fixed window: u16 -> /65535 f32 -> resize f32 -> 3ch
    -> enhance_thermal_fixed_range(normalized=True) (the values are in [0, 1]).  Returns out[3,h,w]."""
    r = ref_preprocess.resize_bilinear(raw_u16.astype(np.float32) / np.float32(65535.0), dst_hw)
    return ref_preprocess.enhance_thermal_fixed_range(np.repeat(r[None], 3, 0), normalized=True)


def golden_frames():
    """The frames oracle/gen_golden.py recorded, regenerated from their seeds; each checked against its raw hash."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "preprocess_kat.npz"))
    raw = np.random.default_rng(0).normal(22800, 400, (512, 640)).clip(0, 65535).astype(np.uint16)
    assert sha(raw) == str(g["raw_sha"])
    night = ref_preprocess.make_raw_frames(3, seed=7)
    frames = {"day0": raw, "mix0": night[0], "mix1": night[1], "mix2": night[2]}
    for name, f in frames.items():
        assert sha(f) == str(g[name + "_raw_sha"]), name
    return g, frames


@pytest.mark.parametrize("name", ["day0", "mix0", "mix1", "mix2"])
def test_fixed_range_paths_reproduce_the_reference(name):
    g, frames = golden_frames()
    for (w, h) in SIZES:
        want = g[f"{name}_{w}x{h}_fixed"]
        assert sha(inference_path_fixed_range(frames[name], (h, w))) == want[0], f"{name} {w}x{h} inference"
        assert sha(train_path_fixed_range(frames[name], (h, w))) == want[1], f"{name} {w}x{h} train"


def test_fixed_range_train_path_holds_raw_counts():
    """The train path's window is applied to raw counts: values of the Freiburg window map to [0, 1]."""
    frame = np.full((8, 10), 23400, np.uint16)
    frame[0, 0] = 0
    out = train_path_fixed_range(frame, (8, 10))
    assert out.shape == (3, 8, 10) and out.dtype == np.float32
    assert out[0, 0, 0] == 0.0 and out[0, 4, 4] == np.float32(0.5)
