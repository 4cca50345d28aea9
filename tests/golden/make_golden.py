#!/usr/bin/env python
"""Generate the golden fixtures in tests/golden/ from the reference's own code path.

Needs torchvision; the ``frames`` case also needs a checkout of the reference
repository for R:im1.png / R:im2.png and is skipped without one:

    python tests/golden/make_golden.py [REFERENCE_REPO_DIR]

What is "the reference" here: RDVC's encoder calls
``torchvision.models.optical_flow.raft_large`` (R:codec_processing.py:48-53,
:1289-1291, :1442), whose ``CorrBlock`` (TV:raft.py:337-431) is the hot path.
The fixtures are outputs of that class on CPU/fp32 (torchvision 0.26.0+cu128,
torch 2.11.0+cu128) for deterministic, RNG-free inputs
(``oracle.corr_numpy.synth_*``), so only outputs need storing.

Fixtures written (each kept under 1 MB; the tests compare full tensors with a
live torchvision run and use these samples to pin that run to the stored one):
  corr_small_odd.npz     (2,32,18,22): odd floor pooling 18x22 -> 9x11 -> 4x5 -> 2x2, B>1.
                         Every ``stride``-th element (5, coprime with every dimension) of
                         the flattened pyramid levels and lookups at sigma 0 / 0.3 / 4 / 40.
  corr_ref_default.npz   (1,256,46,80): RDVC's default RAFT size 368x640
                         (R:codec_processing.py:649-650).  Sampled pyramid entries
                         + strided lookup outputs (full tensors are 72 MB).
  frames_im1_im2.npz     R:im1.png / R:im2.png as uint8 + the stride-4 subsampled
                         final flow of a seed-0 random-init raft_large at 368x640,
                         12 updates, inputs in [0,1] (R:codec_processing.py:751-759).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle import corr_numpy as cn  # noqa: E402
from oracle import tv_corr as tv  # noqa: E402

SIGMAS = (0.0, 0.3, 4.0, 40.0)
SMALL_ODD_STRIDE = 5
REF_DEFAULT_SAMPLES, REF_DEFAULT_STRIDE = 10000, 33


def sample_index(n: int, k: int, seed: int) -> np.ndarray:
    """k deterministic positions in [0, n)."""
    u = cn.hash_uniform(k, seed).astype(np.float64) + 0.5
    return np.minimum((u * n).astype(np.int64), n - 1)


def case_small_odd():
    B, C, h, w = 2, 32, 18, 22
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=3)
    levels = tv.build_pyramid(torch.from_numpy(f1), torch.from_numpy(f2), 4)
    st = SMALL_ODD_STRIDE
    out = {"shape": np.array([B, C, h, w]), "seed": np.array(3), "stride": np.array(st)}
    for l, lv in enumerate(levels):
        out[f"level{l}"] = lv[:, 0].numpy().reshape(-1)[::st].copy()
    for s in SIGMAS:
        co = cn.synth_coords(B, h, w, s, seed=1)
        out[f"lookup_sigma{s:g}"] = tv.index_pyramid(levels, torch.from_numpy(co), 4).numpy().reshape(-1)[::st].copy()
    np.savez_compressed(os.path.join(HERE, "corr_small_odd.npz"), **out)


def case_ref_default():
    B, C, h, w = 1, 256, 46, 80
    f1, f2 = cn.synth_fmaps(B, C, h, w, seed=0)
    levels = tv.build_pyramid(torch.from_numpy(f1), torch.from_numpy(f2), 4)
    out = {"shape": np.array([B, C, h, w]), "seed": np.array(0)}
    for l, lv in enumerate(levels):
        flat = lv.reshape(-1).numpy()
        idx = sample_index(flat.size, REF_DEFAULT_SAMPLES, 77 + l)
        out[f"level{l}_idx"] = idx
        out[f"level{l}_val"] = flat[idx]
    for s in SIGMAS:
        co = cn.synth_coords(B, h, w, s, seed=1)
        o = tv.index_pyramid(levels, torch.from_numpy(co), 4).numpy().reshape(-1)
        out[f"lookup_sigma{s:g}_stride{REF_DEFAULT_STRIDE}"] = o[::REF_DEFAULT_STRIDE].copy()
    np.savez_compressed(os.path.join(HERE, "corr_ref_default.npz"), **out)


def preprocess_frame_raft(frame_u8: np.ndarray, size_hw) -> torch.Tensor:
    """Restates R:codec_processing.py:751-759: to_tensor -> resize(antialias) -> [0,1]."""
    import torchvision.transforms.functional as TF
    t = TF.to_tensor(frame_u8)
    t = TF.resize(t, list(size_hw), antialias=True)
    return t.unsqueeze(0)


def seeded_raft(corr_block=None):
    from torchvision.models.optical_flow import raft_large
    torch.manual_seed(0)
    kw = {} if corr_block is None else {"corr_block": corr_block}
    return raft_large(weights=None, **kw).eval()


def case_frames(ref_dir):
    from PIL import Image
    im1 = np.asarray(Image.open(os.path.join(ref_dir, "im1.png")).convert("RGB"))
    im2 = np.asarray(Image.open(os.path.join(ref_dir, "im2.png")).convert("RGB"))
    a = preprocess_frame_raft(im1, (368, 640))
    b = preprocess_frame_raft(im2, (368, 640))
    model = seeded_raft()
    with torch.no_grad():
        flow = model(a, b, num_flow_updates=12)[-1]
    np.savez_compressed(
        os.path.join(HERE, "frames_im1_im2.npz"),
        im1=im1, im2=im2, flow_stride4=flow[0, :, ::4, ::4].numpy().astype(np.float32),
    )


if __name__ == "__main__":
    case_small_odd()
    case_ref_default()
    if len(sys.argv) > 1:
        case_frames(sys.argv[1])
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))
