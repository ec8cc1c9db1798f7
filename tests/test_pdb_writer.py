"""PDB writer (SURVEY §8(f).2): byte parity with files written by the UNMODIFIED reference (tests/golden/make_golden_pdb.py), the
reference's file-naming rules, and the `analysis.utils` overlay.  Host-only: runs without a GPU."""
import os
import sys

import numpy as np
import pytest

from conftest import golden
from se3_diffusion_b200 import pdb_writer

CASES = ["single_backbone", "traj_mixed", "one_residue_f64"]


@pytest.mark.parametrize("name", CASES)
def test_bytes_equal_reference_writer(name):
    g = golden(f"pdb_{name}")
    got = pdb_writer.format_pdb(g["pos"], aatype=g.get("aatype"), b_factors=g.get("b_factors"))
    exp = g["expected"].tobytes()
    assert len(got) == len(exp), (len(got), len(exp))
    if got != exp:   # point at the first differing line
        gl, el = got.split(b"\n"), exp.split(b"\n")
        k = next(i for i, (a, b) in enumerate(zip(gl, el)) if a != b)
        raise AssertionError(f"line {k}:\n got {gl[k]!r}\n exp {el[k]!r}")


def test_structure_and_edge_cases():
    g = golden("pdb_traj_mixed")
    txt = pdb_writer.format_pdb(g["pos"], aatype=g["aatype"], b_factors=g["b_factors"]).decode()
    lines = txt.split("\n")
    assert lines[-1] == "END" and lines[0].rstrip() == "MODEL     1"
    assert sum(l.startswith("MODEL") for l in lines) == 3 and sum(l.startswith("ENDMDL") for l in lines) == 3
    assert all(len(l) >= 80 for l in lines[:-1])                       # padded, never truncated
    assert any(len(l) > 80 for l in lines)                             # the over-wide coordinates widen their line
    assert " UNK A" in txt and "  -0.000" in txt                       # aatype 20 -> UNK; negative values rounding to zero keep the sign
    with pytest.raises(ValueError):
        pdb_writer.format_pdb(g["pos"], aatype=np.full(9, 21))
    with pytest.raises(ValueError):
        pdb_writer.format_pdb(np.zeros((4, 3)))


def test_file_naming_rules(tmp_path):
    g = golden("pdb_single_backbone")
    d = str(tmp_path)
    p1 = pdb_writer.write_prot_to_pdb(g["pos"], os.path.join(d, "sample.pdb"))
    p2 = pdb_writer.write_prot_to_pdb(g["pos"], os.path.join(d, "sample.pdb"))
    assert os.path.basename(p1) == "sample_1.pdb" and os.path.basename(p2) == "sample_2.pdb"
    p3 = pdb_writer.write_prot_to_pdb(g["pos"], os.path.join(d, "sample.pdb"), overwrite=True)
    assert os.path.basename(p3) == "sample_1.pdb"
    p4 = pdb_writer.write_prot_to_pdb(g["pos"], os.path.join(d, "plain.pdb"), no_indexing=True)
    assert os.path.basename(p4) == "plain.pdb"
    assert open(p4, "rb").read() == g["expected"].tobytes()


def test_overlay_module_next_to_reference(tmp_path):
    """With the overlay ahead of the reference on sys.path, `from analysis import utils` keeps every reference symbol and swaps
    only the writer; both writers produce identical files for a random trajectory."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import ref_harness as rh
    if not rh.reference_available():
        pytest.skip("reference tree not present on this machine")
    rh.install_stubs()
    import importlib.util
    import se3_diffusion_b200
    ov = os.path.join(os.path.dirname(se3_diffusion_b200.__file__), "overlay", "analysis", "utils.py")
    spec = importlib.util.spec_from_file_location("overlay_analysis_utils", ov)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    from analysis import utils as ref_au
    assert mod.write_prot_to_pdb is pdb_writer.write_prot_to_pdb
    assert hasattr(mod, "create_full_prot") and hasattr(mod, "rigids_to_se3_vec")
    rng = np.random.RandomState(0)
    pos = np.zeros((4, 30, 37, 3), np.float32)
    pos[:, :, :5] = (rng.randn(4, 30, 5, 3) * 20).astype(np.float32)
    a = ref_au.write_prot_to_pdb(pos, str(tmp_path / "ref.pdb"), no_indexing=True)
    b = mod.write_prot_to_pdb(pos, str(tmp_path / "ours.pdb"), no_indexing=True)
    assert open(a, "rb").read() == open(b, "rb").read()
    # the way Sampler.save_traj calls it (experiments/inference_se3_diffusion.py:272-287): suffix-less paths, indexed names,
    # b-factors 100 on diffused residues
    bfac = np.tile((np.arange(30) % 3 > 0).astype(float)[:, None] * 100, (1, 37))
    for sub, w in (("r", ref_au.write_prot_to_pdb), ("o", mod.write_prot_to_pdb)):
        d = tmp_path / sub
        d.mkdir()
        p1 = w(pos[0], str(d / "sample"), b_factors=bfac)
        p2 = w(pos, str(d / "bb_traj"), b_factors=bfac)
        p3 = w(pos[0], str(d / "sample"), b_factors=bfac)
        assert [os.path.basename(x) for x in (p1, p2, p3)] == ["sample_1.pdb", "bb_traj_1.pdb", "sample_2.pdb"]
    for fn in ("sample_1.pdb", "bb_traj_1.pdb", "sample_2.pdb"):
        assert open(tmp_path / "r" / fn, "rb").read() == open(tmp_path / "o" / fn, "rb").read()


def test_sampler_calls_write_the_reference_files(tmp_path):
    """Called the way Sampler.save_traj calls the reference's writer (suffix-less paths, indexed names, b-factors 100 on diffused
    residues), the native writer produces the files the unmodified reference wrote for the same trajectory
    (tests/golden/make_golden_overlay.py)."""
    g = golden("pdb_sampler_calls")
    pos, bfac = g["pos"], g["b_factors"]
    plain = pdb_writer.write_prot_to_pdb(pos, str(tmp_path / "ref.pdb"), no_indexing=True)
    assert open(plain, "rb").read() == g["plain"].tobytes()
    paths = [pdb_writer.write_prot_to_pdb(pos[0], str(tmp_path / "sample"), b_factors=bfac),
             pdb_writer.write_prot_to_pdb(pos, str(tmp_path / "bb_traj"), b_factors=bfac),
             pdb_writer.write_prot_to_pdb(pos[0], str(tmp_path / "sample"), b_factors=bfac)]
    assert [os.path.basename(p) for p in paths] == [str(n) for n in g["names"]]
    for p, key in zip(paths, ("sample", "traj", "sample")):
        assert open(p, "rb").read() == g[key].tobytes(), os.path.basename(p)


def test_fixed_point_formatter_equals_printf_on_hard_values():
    """fd_format_pdb's own %8.3f / %6.2f (scale, round-half-even, emit digits; snprintf near ties and beyond 9e15) against Python's
    correctly rounded formatting: float32-born values (exact ties possible), float64 values adjacent to decimal ties, zeros of both
    signs, values that round up into a new digit, huge and tiny magnitudes."""
    rng = np.random.RandomState(3)
    vals = [0.0, -0.0, 0.0005, -0.0005, 0.0015, 0.0025, 999.9995, -999.9995, 9999.9995, 99999.9996, 1e-12, -1e-12, 123456789.125, 1e15,
            0.5 ** 11, 3 * 0.5 ** 11, -5 * 0.5 ** 12, 0.125, 0.375, 2.0625]
    vals += list(rng.randn(3000) * 37.0)
    vals += [float(np.float32(v)) for v in rng.randn(3000) * 37.0]
    ties = (rng.randint(-10 ** 6, 10 ** 6, 2000) + 0.5) / 1000.0          # decimal ties: the nearest doubles lie just above or below
    vals += list(ties) + [float(np.nextafter(t, np.inf)) for t in ties[:500]] + [float(np.nextafter(t, -np.inf)) for t in ties[:500]]
    vals = np.array(vals, dtype=np.float64)
    n = len(vals) // 3 * 3
    pos = np.zeros((1, n // 3, 37, 3))
    pos[0, :, 1, :] = vals[:n].reshape(-1, 3)                               # CA slot
    pos[0, :, 0, 0] = 1.0                                                   # keep residues present even if a CA row is all-zero
    bf = np.zeros((n // 3, 37)); bf[:, 1] = np.abs(vals[:n:3]) % 1000.0
    txt = pdb_writer.format_pdb(pos, b_factors=bf).decode().split("\n")
    ca = [l for l in txt if l.startswith("ATOM") and l[12:16] == " CA "]
    k = 0
    for i in range(n // 3):
        x, y, z = vals[3 * i:3 * i + 3]
        if abs(x) + abs(y) + abs(z) <= 1e-7:
            continue
        want = f"{x:>8.3f}{y:>8.3f}{z:>8.3f}{1.0:>6.2f}{bf[i, 1]:>6.2f}"
        assert ca[k][30:30 + len(want)] == want, (i, x, y, z, ca[k])
        k += 1
    assert k == len(ca)
