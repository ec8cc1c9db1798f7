"""Golden data for the drop-in overlay, produced by the UNMODIFIED reference (its source tree and shipped checkpoints at
FRAMEDIFF_REFERENCE, see ref_harness.py):  python tests/golden/make_golden_overlay.py

state_dict_layout.npz  parameter names and shapes of the reference's ScoreNetwork state_dict and of both shipped checkpoints
                       (weights/{paper,best}_weights.pth, leading 'module.' stripped): what our module must load strict=True
pdb_sampler_calls.npz  the files the reference's write_prot_to_pdb writes for a random trajectory the way Sampler.save_traj calls
                       it (experiments/inference_se3_diffusion.py:272-287), with its inputs
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as rh  # noqa: E402

rh.install_stubs()
from analysis import utils as au  # noqa: E402


def sampler_inputs():
    """4 frames x 30 residues, backbone atoms only, b-factors 100 on diffused residues."""
    rng = np.random.RandomState(0)
    pos = np.zeros((4, 30, 37, 3), np.float32)
    pos[:, :, :5] = (rng.randn(4, 30, 5, 3) * 20).astype(np.float32)
    bfac = np.tile((np.arange(30) % 3 > 0).astype(float)[:, None] * 100, (1, 37))
    return pos, bfac


def layouts():
    out = {}
    net, _ = rh.build_reference()
    sds = {"module": net.state_dict(), "paper_weights": rh.load_reference_checkpoint("paper_weights.pth"),
           "best_weights": rh.load_reference_checkpoint("best_weights.pth")}
    for tag, sd in sds.items():
        out[f"{tag}_names"] = np.array(list(sd))
        shapes = [tuple(v.shape) for v in sd.values()]
        out[f"{tag}_ndim"] = np.array([len(s) for s in shapes], np.int64)
        out[f"{tag}_dims"] = np.array([d for s in shapes for d in s], np.int64)
    np.savez_compressed(os.path.join(HERE, "state_dict_layout.npz"), **out)
    print({k: len(v) for k, v in out.items() if k.endswith("_names")})


def sampler_files():
    pos, bfac = sampler_inputs()
    with tempfile.TemporaryDirectory() as d:
        plain = open(au.write_prot_to_pdb(pos, os.path.join(d, "ref.pdb"), no_indexing=True), "rb").read()
        p1 = au.write_prot_to_pdb(pos[0], os.path.join(d, "sample"), b_factors=bfac)
        p2 = au.write_prot_to_pdb(pos, os.path.join(d, "bb_traj"), b_factors=bfac)
        p3 = au.write_prot_to_pdb(pos[0], os.path.join(d, "sample"), b_factors=bfac)
        names = [os.path.basename(p) for p in (p1, p2, p3)]
        sample, traj, sample2 = (open(p, "rb").read() for p in (p1, p2, p3))
    assert sample == sample2
    np.savez_compressed(os.path.join(HERE, "pdb_sampler_calls.npz"), pos=pos, b_factors=bfac, names=np.array(names),
                        **{k: np.frombuffer(v, np.uint8) for k, v in (("plain", plain), ("sample", sample), ("traj", traj))})
    print(names, len(plain), len(sample), len(traj), "bytes")


if __name__ == "__main__":
    layouts()
    sampler_files()
