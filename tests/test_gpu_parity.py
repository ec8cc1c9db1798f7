"""-m gpu: CUDA path (through the C ABI / the Python host layer) vs the CPU oracle and the reference's golden vectors.

Tolerance (BASELINE.json north_star): bit-exact for indices/masks, 1e-4 relative (max-norm) for fp32 scores and
coordinates.  The IGSO(3) rotation score is only compared where it is well-conditioned (omega <= 3.5 sigma); beyond
that the reference's own mixed fp32/fp64 series is noise-dominated (SURVEY §7.2, tests/test_oracle_golden.py).
"""
import numpy as np
import pytest
import torch

from conftest import assert_close, golden, paper_weights_path, quat_align
from oracle import framediff_oracle as fo

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope="module")
def eng():
    from gpu_common import engine
    return engine("fp32")


def _well_conditioned(t, rigids_t, rigids_pred, k=3.5):
    q = fo.quat_mul(fo.quat_invert(torch.tensor(rigids_pred[..., :4])), torch.tensor(rigids_t[..., :4]).float())
    om = fo.quat_to_rotvec(q).norm(dim=-1).numpy()
    sig = fo.discrete_sigma()[fo.so3_t_to_idx(np.asarray(t, dtype=np.float64))]
    return om <= k * sig[:, None]


def _assert_elementwise(a, b, rtol, name, frac=0.999):
    """north_star: '1e-4 rel ... on scores/coordinates'.  Besides the max-norm bound, elementwise: |a-b| <= rtol*|b| + rtol*rms(b) for at
    least `frac` of the elements and 5x that for every element (a floor tied to the tensor's RMS, not its maximum, so that elements
    far below the maximum are not allowed to be arbitrarily wrong in relative terms)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    nz = b != 0
    rms = float(np.sqrt(np.mean(b[nz] ** 2))) if nz.any() else 0.0
    err = np.abs(a - b)
    bound = rtol * np.abs(b) + rtol * rms
    ok = err <= bound
    assert ok.mean() >= frac, f"{name}: only {ok.mean():.5f} of elements within rtol {rtol:g} (+{rtol:g}*rms {rms:.3g}); worst {err.max():.3e}"
    assert (err <= 5 * bound).all(), f"{name}: {int((err > 5 * bound).sum())} elements beyond 5x the elementwise bound; worst {err.max():.3e}"


def _check_forward(out, ref, t, rigids_t, tol=TOL, name="", psi_tol=None):
    """psi_tol: psi = u/|u| of a 2-vector — where |u| is small the normalisation amplifies the element error of the hidden state, so
    the split-bf16 mode (1e-5 element error) gets 5e-4 on the torsion itself; the O-atom coordinates it places stay under `tol`."""
    o = {k: v.detach().cpu().numpy() for k, v in out.items()}
    for k in ("psi", "trans_score", "atom37", "atom14"):
        assert_close(o[k], ref[k], 0, norm_rel=(psi_tol or tol) if k == "psi" else tol, name=f"{name}{k}")
    for k in ("trans_score", "atom37"):
        _assert_elementwise(o[k], ref[k], tol, name + k + " (elementwise)")
    assert_close(quat_align(o["rigids"][..., :4], ref["rigids"][..., :4]), ref["rigids"][..., :4], 0, atol=20 * tol, name=name + "quat")
    assert_close(o["rigids"][..., 4:], ref["rigids"][..., 4:], 0, norm_rel=tol, name=name + "trans")
    ok = _well_conditioned(t, rigids_t, ref["rigids"])
    assert ok.sum() > 0.4 * ok.size
    assert_close(o["rot_score"][ok], ref["rot_score"][ok], 0, norm_rel=tol, name=name + "rot_score")
    # beyond omega = 3.5 sigma the reference's own series (fp32 terms inside a cancelling fp64 sum) is noise-dominated: an absolute
    # floor instead of silence (SURVEY §7.2) — 2 % of the tensor's largest well-conditioned entry
    if (~ok).any():
        floor = 2e-2 * max(np.abs(ref["rot_score"][ok]).max(), 1e-30)
        bad = np.abs(o["rot_score"][~ok] - ref["rot_score"][~ok]).max()
        assert bad <= floor, f"{name}rot_score (ill-conditioned entries): max|err| {bad:.3e} > floor {floor:.3e}"


# ---- per-residue diffuser kernels -------------------------------------------------------------------------------------
def test_igso3_score_grid(eng):
    g = golden("igso3_score")
    T, W = g["vec"].shape[:2]
    sig = np.repeat(g["sigma"][:, None], W, 1)
    sc = eng.igso3_score(torch.tensor(g["vec"]), torch.tensor(sig)).cpu().numpy()
    om = np.linalg.norm(g["vec"], axis=-1)
    ok = om <= 3.5 * g["sigma"][:, None]
    # elementwise where the reference's own fp32 quotient-rule numerator is not cancellation-dominated (omega >= 0.05) …
    # (relative cancellation of lo*dhi - hi*dlo is ~(l*omega)^2/6, i.e. the reference's fp32 result carries ~1e-3 relative
    # noise at omega = 0.05; elementwise tolerance reflects that, the max-norm check below is the 1e-4 gate)
    mid = ok & (om >= 0.05)
    assert_close(sc[mid], g["score"][mid], 5e-3, atol=1e-6, name="igso3 score (well-conditioned, elementwise)")
    # … and max-norm per sigma row over the whole well-conditioned range (tiny omega: lo*dhi - hi*dlo cancels in fp32
    # in the reference itself, so only the absolute size is meaningful there)
    for r in range(T):
        assert_close(sc[r][mid[r]], g["score"][r][mid[r]], 0, norm_rel=1e-4, name=f"igso3 score row {r}")
        tiny = ok[r] & ~mid[r]      # omega < 0.05: reference value is fp32 cancellation noise; bound the absolute error
        assert_close(sc[r][tiny], g["score"][r][tiny], 0, atol=1e-3 * np.abs(g["score"][r][ok[r]]).max(), name=f"igso3 tiny omega row {r}")
    assert np.all(np.isfinite(sc))


def test_igso3_tables(eng):
    g = golden("schedules")
    idx = [int(fo.so3_t_to_idx(1.0)), int(fo.so3_t_to_idx(0.3))]
    tab = eng.igso3_tables(idx)
    assert_close(tab["cdf"][0], g["cdf_t1"], 1e-9, atol=1e-13, name="cdf(t=1)")
    assert_close(tab["cdf"][1], g["cdf_t03"], 1e-9, atol=1e-13, name="cdf(t=0.3)")
    sel = np.arange(0, 500, 25)
    idxs = [int(fo.so3_t_to_idx(t)) for t in g["t"][sel]]
    assert np.array_equal(np.array(idxs), g["so3_sigma_idx"][sel])
    tab = eng.igso3_tables(idxs)
    assert_close(tab["score_scaling"], g["rot_score_scaling"][sel], 1e-8, name="rot score scaling")
    row = fo.igso3_row(idxs[3])
    assert_close(tab["pdf"][3], row["pdf"], 1e-9, atol=1e-13, name="pdf row")
    assert_close(tab["score_norms"][3], row["score_norms"], 1e-7, atol=1e-9, name="score_norms row")


def test_sample_ref_injected(eng):
    g = golden("sample_ref")
    n = int(g["n"])
    np.random.seed(int(g["seed"]))
    za, ua, zt = np.random.randn(n, 3), np.random.rand(n), np.random.normal(size=(n, 3))
    r = eng.sample_ref(n, za, ua, zt).cpu().numpy()
    assert_close(quat_align(r[:, :4], g["rigids_t"][:, :4]), g["rigids_t"][:, :4], 0, atol=2e-6, name="quat")
    assert_close(r[:, 4:], g["rigids_t"][:, 4:], 1e-6, name="trans")


def test_sample_ref_philox_statistics(eng):
    """Counter-based prior: independent of how the batch is split, right marginals."""
    a = eng.sample_ref(4 * 256, seed=7, first_sample=0, per_sample=256).cpu().numpy()
    b = eng.sample_ref(2 * 256, seed=7, first_sample=2, per_sample=256).cpu().numpy()
    assert np.array_equal(a[512:], b)                     # bit-exact across shardings
    assert abs(np.linalg.norm(a[:, :4], axis=-1) - 1).max() < 1e-6
    tr = a[:, 4:]
    assert abs(tr.mean()) < 1.0 and abs(tr.std() - 10.0) < 0.6
    ang = 2 * np.arccos(np.clip(np.abs(a[:, 0]), 0, 1))
    row = fo.igso3_row(fo.so3_t_to_idx(1.0))
    mean_ref = np.sum(fo.discrete_omega() * row["pdf"]) / np.sum(row["pdf"])
    assert abs(ang.mean() - mean_ref) < 0.08


def test_reverse_step(eng):
    g = golden("reverse_step")
    B, N = g["rigids_t"].shape[:2]
    for j in range(3):
        t, use_mask, center, ns, seed = g[f"cfg_{j}"]
        np.random.seed(int(seed))
        zr, zx = np.random.normal(size=(B, N, 3)), np.random.normal(size=(B, N, 3))
        r, rm = eng.reverse_step(torch.tensor(g["rigids_t"]), g["rot_score"], g["trans_score"], float(t), float(g["dt"]),
                                 diffuse_mask=g["mask"] if use_mask else None, center=bool(center), noise_scale=float(ns),
                                 z_rot=zr, z_trans=zx, want_rotmat=True)
        assert_close(rm.cpu().numpy(), g[f"rot_{j}"], 0, atol=2e-6, name=f"rot_{j}")
        assert_close(r[..., 4:].cpu().numpy(), g[f"trans_{j}"], 0, norm_rel=1e-6, name=f"trans_{j}")
        assert_close(fo.quat_to_rotmat(r[..., :4].cpu()).numpy(), g[f"rot_{j}"], 0, atol=5e-6, name=f"quat_{j}")


def test_reverse_step_rejects_bad_t(eng):
    g = golden("reverse_step")
    with pytest.raises(ValueError):
        eng.reverse_step(torch.tensor(g["rigids_t"]), g["rot_score"], g["trans_score"], 1.5, 0.01)


def test_compute_backbone(eng):
    rs = np.random.RandomState(3)
    q = rs.standard_normal((5, 33, 4)); q /= np.linalg.norm(q, axis=-1, keepdims=True)
    r7 = torch.tensor(np.concatenate([q, rs.standard_normal((5, 33, 3)) * 12], -1), dtype=torch.float32)
    psi = torch.tensor(rs.standard_normal((5, 33, 2)), dtype=torch.float32)
    a37, a14 = eng.compute_backbone(r7, psi)
    r37, mask, r14 = fo.compute_backbone(fo.quat_to_rotmat(r7[..., :4]), r7[..., 4:], psi)
    assert_close(a37.cpu().numpy(), r37.numpy(), 0, norm_rel=1e-6, name="atom37")
    assert_close(a14.cpu().numpy(), r14.numpy(), 0, norm_rel=1e-6, name="atom14")
    assert np.array_equal(np.any(a37.cpu().numpy() != 0, axis=-1), mask.numpy())   # atom37 mask: bit-exact


# ---- ScoreNetwork.forward -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("idx", [0, 1, 2, 3])
def test_forward_golden_fp32(eng, idx):
    """CUDA forward vs the UNMODIFIED reference's outputs (synthetic weights; padded + fixed-mask + ragged N cases)."""
    from gpu_common import feats_from_golden
    g = golden(f"forward_synth_{idx}")
    out = eng.forward(feats_from_golden(g))
    ref = {k[4:]: v for k, v in g.items() if k.startswith("out_")}
    for k in ("rot_score", "trans_score", "psi", "rigids", "atom37"):
        assert out[k].dtype == torch.tensor(ref[k]).dtype, f"{k}: dtype {out[k].dtype}"
    _check_forward(out, ref, g["in_t"], g["in_rigids_t"])


def test_forward_intermediates_vs_oracle(eng):
    """Stage-by-stage taps vs the oracle's trace (localises a regression to a kernel)."""
    from gpu_common import feats_from_golden
    g = golden("forward_synth_1")
    f = feats_from_golden(g)
    B, N = f["rigids_t"].shape[:2]
    eng.set_debug(True)
    try:
        eng.forward(f)
        trace = {}
        with torch.no_grad():
            fo.score_network_forward(fo.as_torch_weights(fo.synthetic_weights(0)), f, trace=trace)
        assert_close(eng.debug_fetch("node_embed", (B, N, 256)), trace["node_embed"].numpy(), 0, norm_rel=2e-5, name="node_embed")
        assert_close(eng.debug_fetch("edge_embed", (B, N, N, 128)), trace["edge_embed"].numpy(), 0, norm_rel=2e-5, name="edge_embed")
        Np = (N + 3) // 4 * 4
        for b in range(4):
            att = eng.debug_fetch(f"attn_{b}", (B, 8, N, Np))[..., :N]
            # padded QUERY rows sit at logits ~ -1e5 (fp32 ulp 0.008): their softmax is rounding noise in the reference
            # too and is multiplied by the mask downstream — compare valid query rows only
            valid = (f["res_mask"].numpy() > 0.5)[:, None, :, None]
            assert_close(att * valid, trace[f"attn_{b}"].numpy() * valid, 0, atol=2e-5 * (b + 1), name=f"attn_{b}")
            assert_close(eng.debug_fetch(f"ipa_feats_{b}", (B, N, 2688)), trace[f"ipa_feats_{b}"].numpy(), 0, norm_rel=5e-5, name=f"ipa_feats_{b}")
            assert_close(eng.debug_fetch(f"node_{b}", (B, N, 256)), trace[f"node_{b}"].numpy(), 0, norm_rel=5e-5, name=f"node_{b}")
            assert_close(eng.debug_fetch(f"trans_{b}", (B, N, 3)), trace[f"trans_{b}"].numpy(), 0, norm_rel=5e-5, name=f"trans_{b}")
            if b < 3:
                assert_close(eng.debug_fetch(f"edge_{b}", (B, N, N, 128)), trace[f"edge_{b}"].numpy(), 0, norm_rel=5e-5, name=f"edge_{b}")
    finally:
        eng.set_debug(False)


def test_forward_vs_oracle_larger(eng):
    """B=2, N=96 (several GEMM tiles, N not a multiple of 64), random masks: CUDA vs oracle on the same inputs."""
    np.random.seed(5)
    B, N = 2, 96
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.8, 0.62], dtype=torch.float64)
    f["sc_ca_t"] = torch.tensor(np.random.randn(B, N, 3) * 9)
    f["res_mask"][1, 80:] = 0
    f["seq_idx"][1, 80:] = 0
    f["fixed_mask"][0, 10:20] = 1
    f["torsion_angles_sin_cos"] = torch.tensor(np.random.randn(B, N, 7, 2))
    with torch.no_grad():
        ref = fo.score_network_forward(fo.as_torch_weights(fo.synthetic_weights(0)), f)
    out = eng.forward(f)
    _check_forward(out, {k: v.numpy() for k, v in ref.items()}, f["t"].numpy(), f["rigids_t"].numpy())


def test_forward_se3_equivariance(eng):
    """Size-independent property: a global rotation+translation of the input frames leaves scores in the local frame
    unchanged: trans_score rotates, psi invariant, predicted frames move rigidly.  N=160, B=3."""
    np.random.seed(9)
    B, N = 3, 160
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.9, 0.7, 0.5], dtype=torch.float64)
    out1 = eng.forward(f)
    qg = torch.tensor([0.3, -0.5, 0.1, 0.8], dtype=torch.float32); qg /= qg.norm()
    Rg = fo.quat_to_rotmat(qg)
    tg = torch.tensor([3.0, -7.0, 11.0])
    f2 = dict(f)
    q_new = fo.quat_mul(qg.expand(B, N, 4), r7[..., :4])
    x_new = fo.rot_apply(Rg, r7[..., 4:]) + tg
    f2["rigids_t"] = torch.cat([q_new, x_new], -1)
    out2 = eng.forward(f2)
    a1 = out1["atom37"].cpu(); a2 = out2["atom37"].cpu()
    moved = fo.rot_apply(Rg, a1) + tg
    nz = (a1.abs().sum(-1, keepdim=True) > 0).float()
    # translation invariance is only approximate in the reference model itself (global coordinates enter the IPA
    # point features) — compare the rotation-only part exactly and the full transform loosely
    assert_close(out2["psi"].cpu().numpy(), out1["psi"].cpu().numpy(), 0, atol=5e-3, name="psi invariance")
    assert_close((a2 * nz).numpy(), (moved * nz).numpy(), 0, norm_rel=5e-3, name="atom37 equivariance")


def test_forward_batch_consistency(eng):
    """A sample's outputs do not depend on what else is in the batch (no cross-sample op on the path)."""
    np.random.seed(11)
    N = 64
    r7 = torch.stack([fo.sample_ref(N) for _ in range(3)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.9, 0.7, 0.5], dtype=torch.float64)
    full = eng.forward(f)
    one = eng.forward({k: v[1:2] for k, v in f.items()})
    for k in ("trans_score", "psi", "rigids"):
        assert_close(one[k].cpu().numpy(), full[k][1:2].cpu().numpy(), 0, norm_rel=1e-5, name=k)


# ---- the reverse loop (Experiment.inference_fn) ---------------------------------------------------------------------------
def test_trajectory_vs_reference_golden(eng):
    """Engine loop with the reference's numpy noise injected vs the reference's real inference_fn (golden)."""
    from gpu_common import numpy_noise
    g = golden("traj_synth")
    B, N, num_t = int(g["B"]), int(g["N"]), int(g["num_t"])
    noise = numpy_noise(int(g["seed"]), B, N, num_t)
    out = eng.sample(B, N, num_t=num_t, min_t=0.01, noise_scale=float(g["noise_scale"]), aux_traj=True, noise=noise, use_graph=True)
    assert out["prot_traj"].shape == g["prot_traj"].shape and out["rigid_traj"].shape == g["rigid_traj"].shape
    # prior
    assert_close(out["rigid_traj"][-1][..., 4:], g["rigid_traj"][-1][..., 4:], 1e-6, name="prior trans")
    # first reverse step (index -2 after the reference's flip) — tight
    assert_close(out["rigid_traj"][-2][..., 4:], g["rigid_traj"][-2][..., 4:], 0, norm_rel=TOL, name="step-1 trans")
    assert_close(out["prot_traj"][-1], g["prot_traj"][-1], 0, norm_rel=TOL, name="step-1 atom37")
    assert_close(out["rigid_0_traj"][-1], g["rigid_0_traj"][-1], 0, norm_rel=TOL, name="step-1 x0 atom37")
    assert_close(out["trans_traj"][-1], g["trans_traj"][-1], 0, norm_rel=TOL, name="step-1 trans_traj")


def test_trajectory_motif_scaffolding_masks_vs_oracle(eng):
    """SURVEY §8(f).3: fixed (motif) residues and padded positions through the whole loop — rigids_init given, fixed_mask on a segment,
    res_mask with trailing padding, noise injected; engine loop vs the oracle's restatement of inference_fn, step by step."""
    np.random.seed(5)
    B, N, num_t = 2, 40, 6
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["res_mask"] = torch.ones(B, N, dtype=torch.float64); f["res_mask"][1, 33:] = 0.0
    f["fixed_mask"] = torch.zeros(B, N, dtype=torch.float64); f["fixed_mask"][:, 10:18] = 1.0
    f["seq_idx"] = (torch.arange(1, N + 1)[None].repeat(B, 1) * f["res_mask"].long()).long()
    tors = np.random.randn(B, N, 7, 2); tors /= np.linalg.norm(tors, axis=-1, keepdims=True)
    f["torsion_angles_sin_cos"] = torch.tensor(tors)          # the psi imputed on the motif residues (non-zero: places their O atoms)
    zr = np.random.normal(size=(num_t - 1, B, N, 3)); zx = np.random.normal(size=(num_t - 1, B, N, 3))
    ref = fo.inference_loop(fo.as_torch_weights(fo.synthetic_weights(0)), f, num_t=num_t, min_t=0.01, aux_traj=True, noise_scale=0.5,
                            noise_fn=lambda step, shape: (zr[step], zx[step]))
    out = eng.sample(B, N, num_t=num_t, min_t=0.01, noise_scale=0.5, aux_traj=True, use_graph=True, rigids_init=r7,
                     noise={"z_rot": zr, "z_trans": zx}, res_mask=f["res_mask"], fixed_mask=f["fixed_mask"], seq_idx=f["seq_idx"],
                     gt_psi=tors[:, :, 2, :])
    assert_close(out["psi_pred"][0][fixed_idx := (f["fixed_mask"].numpy() > 0.5)], tors[:, :, 2, :][fixed_idx], 1e-6, name="imputed psi")
    # fixed residues never move; diffused ones follow the oracle (first reverse step tight, last frame looser: error compounds)
    fixed = f["fixed_mask"].numpy().astype(bool) & f["res_mask"].numpy().astype(bool)
    got, init = out["rigid_traj"][0][fixed], r7.numpy()[fixed]
    assert np.allclose(got[:, 4:], init[:, 4:], atol=1e-5)                           # translations untouched (not even re-centred)
    assert np.all(np.abs(np.sum(got[:, :4] * init[:, :4], -1)) > 1 - 1e-6)            # same rotation (quaternion up to sign / rounding)
    assert_close(out["rigid_traj"][-2][..., 4:], ref["rigid_traj"][-2][..., 4:], 0, norm_rel=TOL, name="step-1 trans")
    assert_close(out["prot_traj"][-1], ref["prot_traj"][-1], 0, norm_rel=TOL, name="step-1 atom37")
    assert_close(out["prot_traj"][0], ref["prot_traj"][0], 0, norm_rel=2e-3, name="final atom37")


def test_trajectory_graph_equals_eager(eng):
    from gpu_common import numpy_noise
    B, N, num_t = 2, 40, 6
    noise = numpy_noise(3, B, N, num_t)
    a = eng.sample(B, N, num_t=num_t, aux_traj=True, noise=noise, use_graph=True)
    b = eng.sample(B, N, num_t=num_t, aux_traj=True, noise=noise, use_graph=False)
    for k in ("prot_traj", "rigid_traj", "trans_traj", "rigid_0_traj"):
        assert np.array_equal(a[k], b[k]), k          # same kernels, same order: bit-exact
    assert a["kernel_launches"] == b["kernel_launches"] > 0


def test_trajectory_philox_sharding_invariance(eng):
    """Multi-GPU contract (SURVEY §8e): sample g's trajectory depends only on (seed, g), not on the batch it is in."""
    N, num_t = 48, 5
    full = eng.sample(4, N, num_t=num_t, seed=99, first_sample=0)
    part = eng.sample(2, N, num_t=num_t, seed=99, first_sample=2)
    assert_close(part["prot_traj"][0], full["prot_traj"][0][2:], 0, norm_rel=1e-5, name="sharded == full")
    ca = full["prot_traj"][0][:, :, 1]
    assert np.all(np.isfinite(ca))


@pytest.mark.skipif(paper_weights_path() is None, reason="paper_weights.npz not available")
def test_paper_weights_forward_and_config1():
    """BASELINE config 1 (1 x N=60 x 50 steps, paper weights): CUDA loop vs the reference's inference_fn golden."""
    from gpu_common import engine, feats_from_golden, numpy_noise
    e = engine("fp32", weights=paper_weights_path())
    g = golden("forward_paper_0")
    out = e.forward(feats_from_golden(g))
    ref = {k[4:]: v for k, v in g.items() if k.startswith("out_")}
    assert_close(out["rot_score"][0, 0].cpu().numpy(), [0.0447965874, 0.2275690462, -0.2102767425], 1e-4, name="KAT rot")   # SURVEY §8(c)
    assert_close(out["trans_score"][0, 0].cpu().numpy(), [1.5382335178, -0.0656681920, -0.1524047544], 1e-4, name="KAT trans")
    _check_forward(out, ref, g["in_t"], g["in_rigids_t"])
    g = golden("traj_paper_c1")
    noise = numpy_noise(int(g["seed"]), 1, 60, 50)
    out = e.sample(1, 60, num_t=50, min_t=0.01, noise_scale=0.1, aux_traj=True, noise=noise)
    assert_close(out["prot_traj"][0], g["prot_final"], 0, norm_rel=2e-4, name="config-1 final atom37")
    ca = out["prot_traj"][0][0, :, 1]
    assert abs(np.linalg.norm(ca[1:] - ca[:-1], axis=-1).mean() - 3.8088) < 5e-3


# ---- the benchmarked shapes against the ORACLE (not the engine against itself) -------------------------------------------------
@pytest.mark.parametrize("prec,B,N", [("fp32", 2, 128), ("bf16x3", 2, 128), ("fp32", 1, 256), ("bf16x3", 1, 256), ("fp32", 1, 384),
                                      ("bf16x3", 1, 384)])
def test_forward_vs_oracle_bench_shapes(prec, B, N):
    """BASELINE configs 2/3/5: N = 128, 256 (the bench shape) and 384 (> 256: the two-kernel IPA edge path), masks on, non-zero
    self-conditioning and torsions — CUDA (both the CUDA-core fp32 mode and the tcgen05 bf16x3 mode) vs the CPU oracle."""
    from gpu_common import engine
    np.random.seed(100 + N)
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.83, 0.41][:B], dtype=torch.float64)
    f["sc_ca_t"] = torch.tensor(np.random.randn(B, N, 3) * 9)
    f["res_mask"][B - 1, N - 17:] = 0
    f["seq_idx"][B - 1, N - 17:] = 0
    f["fixed_mask"][0, 20:33] = 1
    f["torsion_angles_sin_cos"] = torch.tensor(np.random.randn(B, N, 7, 2))
    with torch.no_grad():
        ref = fo.score_network_forward(fo.as_torch_weights(fo.synthetic_weights(0)), f)
    out = engine(prec).forward(f)
    _check_forward(out, {k: v.numpy() for k, v in ref.items()}, f["t"].numpy(), f["rigids_t"].numpy(), name=f"{prec} B{B} N{N} ",
                   psi_tol=None if prec == "fp32" else 5e-4)


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_trajectory_final_frame_vs_reference_golden(prec):
    """All 12 steps of the reference's own inference_fn run (golden): the final frame, not only the first step.  The per-step error
    (1e-5 relative) compounds through the stochastic loop, hence the looser bound."""
    from gpu_common import engine, numpy_noise
    g = golden("traj_synth")
    B, N, num_t = int(g["B"]), int(g["N"]), int(g["num_t"])
    noise = numpy_noise(int(g["seed"]), B, N, num_t)
    out = engine(prec).sample(B, N, num_t=num_t, min_t=0.01, noise_scale=float(g["noise_scale"]), aux_traj=True, noise=noise)
    assert_close(out["prot_traj"][0], g["prot_traj"][0], 0, norm_rel=2e-3, name="final atom37")
    assert_close(out["rigid_traj"][0][..., 4:], g["rigid_traj"][0][..., 4:], 0, norm_rel=2e-3, name="final trans")
    mid = num_t // 2
    assert_close(out["prot_traj"][mid], g["prot_traj"][mid], 0, norm_rel=1e-3, name="mid-trajectory atom37")


def _kabsch_rmsd(a, b):
    a, b = a - a.mean(0), b - b.mean(0)
    u, s, vt = np.linalg.svd(a.T @ b)
    d = np.sign(np.linalg.det(u @ vt))
    return float(np.sqrt(max((a ** 2).sum() + (b ** 2).sum() - 2 * (s[0] + s[1] + d * s[2]), 0.0) / len(a)))


@pytest.mark.skipif(paper_weights_path() is None, reason="paper_weights.npz not available")
def test_500_step_sampling_statistics_bf16x3_vs_fp32():
    """SURVEY §7.2: the tensor-core mode over a full 500-step sampling with the shipped checkpoint — chain geometry (mean consecutive
    CA-CA 3.80 +- 0.05 A in both modes) and drift against the fp32 engine on the same Philox noise (aligned CA RMSD)."""
    from gpu_common import engine
    res = {}
    for prec in ("fp32", "bf16x3"):
        e = engine(prec, weights=paper_weights_path())
        res[prec] = e.sample(2, 60, num_t=500, min_t=0.01, noise_scale=0.1, seed=321)["prot_traj"][0][:, :, 1]
    for prec, ca in res.items():
        d = np.linalg.norm(ca[:, 1:] - ca[:, :-1], axis=-1)
        assert abs(d.mean() - 3.80) < 0.05, f"{prec}: mean CA-CA {d.mean():.4f}"
    for b in range(2):
        rmsd = _kabsch_rmsd(res["fp32"][b], res["bf16x3"][b])
        assert rmsd < 1.0, f"sample {b}: bf16x3 drifted {rmsd:.3f} A (CA RMSD) from the fp32 engine over 500 steps"


def test_philox_step_noise_moments(eng):
    """The on-device step noise (Philox + Box-Muller) is standard normal: one reverse step with zero scores isolates it."""
    B, N = 4, 256
    r7 = torch.zeros(B, N, 7); r7[..., 0] = 1.0
    zero = np.zeros((B, N, 3))
    t, dt = 0.5, 0.002
    out, _ = eng.reverse_step(r7, zero, zero, t, dt, center=False, noise_scale=1.0, seed=17, first_sample=0, step=3)
    x = out[..., 4:].double().cpu().numpy() * 0.1          # x' = x - (f dt + g sqrt(dt) z) with x = 0  ->  -g sqrt(dt) z
    g_t = np.sqrt(fo.r3_b_t(t))
    z = -x / (g_t * np.sqrt(dt))
    assert abs(z.mean()) < 0.06 and abs(z.std() - 1.0) < 0.04
    assert abs(np.mean(z ** 3)) < 0.15 and abs(np.mean(z ** 4) - 3.0) < 0.3
    # rotation noise: rotvec of the step = g sqrt(dt) z_rot (score 0)
    ang = 2 * np.arccos(np.clip(np.abs(out[..., 0].double().cpu().numpy()), 0, 1))
    zr = ang / (fo.so3_diffusion_coef(t) * np.sqrt(dt))     # |z_rot| ~ chi(3): mean 2 sqrt(2/pi)
    assert abs(zr.mean() - 2 * np.sqrt(2 / np.pi)) < 0.06


def test_diffuser_api_score_on_gpu(eng):
    """SURVEY row a24: SE3Diffuser.score through the mirror class on the device vs the reference's golden (fp64 numpy `score` there;
    the mixed-precision torch_score kernel here — compared where the series is well-conditioned, floor elsewhere)."""
    from se3_diffusion_b200.se3_diffuser import SE3Diffuser
    g = golden("forward_marginal")
    dif = SE3Diffuser(_conf()[1])
    dif.bind_engine(eng)
    ts, rs = dif.score(torch.tensor(g["rigids_0"]), torch.tensor(g["rigids_1"]), float(g["score_t"]))
    assert_close(ts, g["score_trans"], 1e-6, atol=1e-9, name="score trans")
    assert np.asarray(rs).shape == g["score_rot"].shape          # incl. the reference's leading broadcast dimension
    rs, g = np.asarray(rs).reshape(-1, 3), dict(g, score_rot=g["score_rot"].reshape(-1, 3))
    sig = fo.discrete_sigma()[fo.so3_t_to_idx(float(g["score_t"]))]
    om = np.linalg.norm(fo._rotvec_from_quat7(torch.tensor(g["rigids_1"]))[1], axis=-1)
    ok = om <= 3.5 * sig
    assert ok.sum() > 0.3 * ok.size
    assert_close(np.asarray(rs)[ok], g["score_rot"][ok], 0, norm_rel=1e-4, name="score rot (well-conditioned)")
    if (~ok).any():
        assert np.abs(np.asarray(rs)[~ok] - g["score_rot"][~ok]).max() <= 2e-2 * np.abs(g["score_rot"][ok]).max()


# ---- tensor-core (tcgen05) precisions ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("idx", [0, 1, 2, 3])
def test_forward_golden_bf16x3(idx):
    """3-term split-bf16 tensor-core mode must meet the same 1e-4 bar as fp32 (vs the UNMODIFIED reference's outputs)."""
    from gpu_common import engine, feats_from_golden
    e = engine("bf16x3")
    g = golden(f"forward_synth_{idx}")
    out = e.forward(feats_from_golden(g))
    ref = {k[4:]: v for k, v in g.items() if k.startswith("out_")}
    _check_forward(out, ref, g["in_t"], g["in_rigids_t"])


def test_forward_intermediates_bf16x3():
    from gpu_common import engine, feats_from_golden
    e = engine("bf16x3")
    g = golden("forward_synth_2")
    f = feats_from_golden(g)
    B, N = f["rigids_t"].shape[:2]
    e.set_debug(True)
    try:
        e.forward(f)
        trace = {}
        with torch.no_grad():
            fo.score_network_forward(fo.as_torch_weights(fo.synthetic_weights(0)), f, trace=trace)
        assert_close(e.debug_fetch("edge_embed", (B, N, N, 128)), trace["edge_embed"].numpy(), 0, norm_rel=4e-5, name="edge_embed")
        for b in range(3):
            assert_close(e.debug_fetch(f"edge_{b}", (B, N, N, 128)), trace[f"edge_{b}"].numpy(), 0, norm_rel=6e-5, name=f"edge_{b}")
    finally:
        e.set_debug(False)


def test_forward_golden_bf16_throughput_mode():
    """Single-pass bf16 is the throughput mode: documented accuracy ~1e-3 (not the parity mode); checked against a looser bar."""
    from gpu_common import engine, feats_from_golden
    e = engine("bf16")
    g = golden("forward_synth_2")
    out = e.forward(feats_from_golden(g))
    ref = {k[4:]: v for k, v in g.items() if k.startswith("out_")}
    _check_forward(out, ref, g["in_t"], g["in_rigids_t"], tol=2e-2)


def test_trajectory_bf16x3_vs_reference_golden():
    from gpu_common import engine, numpy_noise
    e = engine("bf16x3")
    g = golden("traj_synth")
    B, N, num_t = int(g["B"]), int(g["N"]), int(g["num_t"])
    noise = numpy_noise(int(g["seed"]), B, N, num_t)
    out = e.sample(B, N, num_t=num_t, min_t=0.01, noise_scale=float(g["noise_scale"]), aux_traj=True, noise=noise, use_graph=True)
    assert_close(out["rigid_traj"][-2][..., 4:], g["rigid_traj"][-2][..., 4:], 0, norm_rel=TOL, name="step-1 trans")
    assert_close(out["prot_traj"][-1], g["prot_traj"][-1], 0, norm_rel=TOL, name="step-1 atom37")


def test_tensor_core_large_tile_counts():
    """More row tiles than SMs and a ragged last tile (E = 2*150*150 = 45000 rows = 351.6 tiles): bf16x3 vs fp32 engine."""
    from gpu_common import engine
    np.random.seed(21)
    B, N = 2, 150
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.75, 0.55], dtype=torch.float64)
    f["sc_ca_t"] = torch.tensor(np.random.randn(B, N, 3) * 9)
    e = engine("fp32")
    ref = {k: v.cpu().numpy() for k, v in e.forward(f).items()}
    e = engine("bf16x3")
    out = e.forward(f)
    _check_forward(out, ref, f["t"].numpy(), f["rigids_t"].numpy())


def test_tensor_core_chain_longer_than_256():
    """N > 256 takes the two-kernel IPA edge path (pair-bias GEMM + attention kernel, K = 256 logits GEMM): bf16x3 vs fp32 engine."""
    from gpu_common import engine
    np.random.seed(22)
    B, N = 1, 272
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.35], dtype=torch.float64)
    f["sc_ca_t"] = torch.tensor(np.random.randn(B, N, 3) * 12)
    e = engine("fp32")
    ref = {k: v.cpu().numpy() for k, v in e.forward(f).items()}
    e = engine("bf16x3")
    out = e.forward(f)
    _check_forward(out, ref, f["t"].numpy(), f["rigids_t"].numpy())


def test_cross_check_paths_match_oracle():
    """FD_TC_UNFUSED=1 (EdgeTransition as three GEMM launches), FD_IPA_EDGE2=1 (two-kernel IPA edge pass) and FD_TF_ATTN_GEMM=1
    (sequence attention as batched GEMMs + softmax) are kept as independent implementations of the fused kernels: they must meet the
    same bars.  The switches are read at handle creation,
    so the checks run in a child interpreter."""
    import os, subprocess, sys
    env = dict(os.environ, FD_TC_UNFUSED="1", FD_IPA_EDGE2="1", FD_TF_ATTN_GEMM="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", "-k",
                        "test_forward_golden_bf16x3 or test_forward_intermediates_bf16x3"], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]
    # experimental switch: the fused EdgeTransition as 2-CTA clusters sharing every weight block through TMA multicast
    env = dict(os.environ, FD_TC_CLUSTER="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", "-k",
                        "test_forward_golden_bf16x3 or test_tensor_core_large_tile_counts"], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]


# ---- reference-facing host API (se3_diffusion_b200.se3_diffuser.SE3Diffuser / score_network.ScoreNetwork) -------------------
def _conf():
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import ref_harness as rh
    return rh.default_conf()


def test_diffuser_api_forward_marginal_and_scalings(eng):
    """SE3Diffuser.forward_marginal through the mirror class, numpy RNG seeded like the reference run that made the golden."""
    from se3_diffusion_b200.se3_diffuser import SE3Diffuser
    g = golden("forward_marginal")
    dif = SE3Diffuser(_conf()[1])
    dif.bind_engine(eng)
    for j in range(2):
        t, use_mask, seed = g[f"cfg_{j}"]
        np.random.seed(int(seed))
        o = dif.forward_marginal(torch.tensor(g["rigids_0"]), float(t), diffuse_mask=g["mask"] if use_mask else None, as_tensor_7=True)
        assert_close(fo.quat_to_rotmat(o["rigids_t"][..., :4]).numpy(), g[f"rot_{j}"], 0, atol=5e-6, name="rot_t")
        assert_close(o["rigids_t"][..., 4:].numpy(), g[f"trans_{j}"], 0, norm_rel=2e-6, name="trans_t")
        assert_close(o["trans_score"], g[f"trans_score_{j}"], 1e-7, atol=1e-9, name="trans_score")
        om = np.linalg.norm(g[f"rot_score_{j}"], axis=-1)
        assert_close(o["rot_score"], g[f"rot_score_{j}"], 0, norm_rel=1e-4, name="rot_score")
        assert_close([o["trans_score_scaling"], o["rot_score_scaling"]], g[f"scal_{j}"], 1e-8, name="scalings")
    gs = golden("schedules")
    for k in (0, 137, 499):
        rot, tr = dif.score_scaling(float(gs["t"][k]))
        assert_close([rot, tr], [gs["rot_score_scaling"][k], gs["trans_score_scaling"][k]], 1e-8, name="score_scaling")
    with pytest.raises(ValueError):
        dif.score_scaling(1.5)


def test_diffuser_api_reverse_and_sample_ref_follow_numpy_rng(eng):
    from se3_diffusion_b200.se3_diffuser import SE3Diffuser
    dif = SE3Diffuser(_conf()[1])
    dif.bind_engine(eng)
    g = golden("sample_ref")
    np.random.seed(int(g["seed"]))
    r = dif.sample_ref(int(g["n"]), as_tensor_7=True)["rigids_t"].numpy()
    assert_close(quat_align(r[:, :4], g["rigids_t"][:, :4]), g["rigids_t"][:, :4], 0, atol=2e-6, name="sample_ref quat")
    assert_close(r[:, 4:], g["rigids_t"][:, 4:], 1e-6, name="sample_ref trans")
    g = golden("reverse_step")
    for j in range(3):
        t, use_mask, center, ns, seed = g[f"cfg_{j}"]
        np.random.seed(int(seed))
        out = dif.reverse(torch.tensor(g["rigids_t"]), g["rot_score"], g["trans_score"], float(t), float(g["dt"]),
                          diffuse_mask=g["mask"] if use_mask else None, center=bool(center), noise_scale=float(ns))
        out = out.to_tensor_7() if hasattr(out, "to_tensor_7") else out
        assert_close(fo.quat_to_rotmat(out[..., :4].float().cpu()).numpy(), g[f"rot_{j}"], 0, atol=5e-6, name=f"reverse rot {j}")
        assert_close(out[..., 4:].cpu().numpy(), g[f"trans_{j}"], 0, norm_rel=1e-6, name=f"reverse trans {j}")
    with pytest.raises(ValueError):
        dif.sample_ref(4, diffuse_mask=np.ones(4))          # "Must provide imputation values."


def test_score_network_module_forward_matches_reference_golden():
    """The nn.Module mirror (what the reference's Experiment wraps): state_dict in, reference-shaped dict out."""
    from gpu_common import feats_from_golden, synthetic_state
    from se3_diffusion_b200.score_network import ScoreNetwork
    from se3_diffusion_b200.se3_diffuser import SE3Diffuser
    mc, dc = _conf()
    net = ScoreNetwork(mc, SE3Diffuser(dc), precision="bf16x3")
    net.load_state_dict({k: torch.tensor(v) for k, v in synthetic_state(0).items()}, strict=True)
    net = net.to("cuda").eval()
    g = golden("forward_synth_1")
    f = {k: v.to("cuda") for k, v in feats_from_golden(g).items()}
    with torch.no_grad():
        out = net(f)
    assert set(out) == {"psi", "rot_score", "trans_score", "rigids", "atom37", "atom14"}
    ref = {k[4:]: v for k, v in g.items() if k.startswith("out_")}
    _check_forward(out, ref, g["in_t"], g["in_rigids_t"])
    # train() mode without autograd (the self-conditioning forward inside loss_fn): torch's TransformerEncoder is off its fused path there,
    # i.e. the float key-padding mask is added to the logits — the training-mode CUDA forward; equals the oracle with float_mask_quirk
    net.train()
    with torch.no_grad():
        out_t = net(f)
        ref_t = fo.score_network_forward(fo.as_torch_weights(synthetic_state(0)), feats_from_golden(g), float_mask_quirk=True)
    _check_forward(out_t, {k: v.numpy() for k, v in ref_t.items()}, g["in_t"], g["in_rigids_t"])


def test_inference_fn_numpy_noise_matches_reference_golden(eng):
    """Engine.inference_fn = Experiment.inference_fn: same np.random stream, same return dict, vs the reference run."""
    g = golden("traj_synth")
    B, N, num_t = int(g["B"]), int(g["N"]), int(g["num_t"])
    np.random.seed(int(g["seed"]))
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])       # the caller draws the prior exactly like Sampler.sample
    data = fo.init_feats(r7)
    out = eng.inference_fn(data, num_t=num_t, min_t=0.01, aux_traj=True, noise_scale=float(g["noise_scale"]), noise="numpy")
    for k in ("prot_traj", "rigid_traj", "trans_traj", "rigid_0_traj"):
        assert out[k].shape == g[k].shape, k
    assert tuple(out["psi_pred"].shape) == tuple(g["psi_pred"].shape)
    assert_close(out["prot_traj"][-1], g["prot_traj"][-1], 0, norm_rel=TOL, name="step-1 atom37")
    assert_close(out["rigid_traj"][-2][..., 4:], g["rigid_traj"][-2][..., 4:], 0, norm_rel=TOL, name="step-1 trans")


@pytest.mark.parametrize("tag", ["a", "b"])
def test_loss_forward_vs_reference_loss_fn(eng, tag):
    """SURVEY row a27 (forward half): fd_loss_forward on the reference's own batch and model outputs vs the values its real
    Experiment.loss_fn produced (golden), every term per sample; and end to end from our forward of the same batch."""
    g = golden(f"loss_{tag}")
    batch = {k[3:]: v for k, v in g.items() if k.startswith("in_")}
    mo = {k[4:]: v for k, v in g.items() if k.startswith("out_")}
    got = eng.loss_forward(mo, batch)
    for k in ("batch_rot_loss", "batch_trans_loss", "batch_bb_atom_loss", "batch_dist_mat_loss", "batch_train_loss", "total_loss", "rot_loss",
              "trans_loss", "bb_atom_loss", "dist_mat_loss"):
        assert_close(got[k].cpu().numpy(), g["aux_" + k], 2e-6, atol=1e-9, name=k)
    # the same loss from OUR forward of the batch (fp32 engine): model parity (1e-4) carries through to the loss
    f = {k: torch.as_tensor(batch[k]) for k in ("rigids_t", "res_mask", "fixed_mask", "seq_idx", "t", "sc_ca_t", "torsion_angles_sin_cos")}
    ours = eng.forward(f)
    got2 = eng.loss_forward(ours, batch)
    assert_close(got2["batch_train_loss"].cpu().numpy(), g["aux_batch_train_loss"], 5e-4, name="loss from our forward")


# ---- SURVEY §8(f) rows 1 and 4: batched training-data assembly and eval metrics on the device -------------------------------------------
def test_forward_marginal_batch_padded_vs_single_and_oracle(eng):
    """fd_forward_marginal_batch (one call for a padded batch, per-example t) == the per-example kernel on the unpadded chains, zeros on the
    padding (du.pad_feats), and the oracle's forward_marginal on one of them."""
    rs = np.random.RandomState(8)
    B, N = 3, 40
    lens = [40, 33, 21]
    ts = [0.7, 0.31, 0.05]
    r0 = np.zeros((B, N, 7), np.float32); mask = np.zeros((B, N), np.float32)
    za, ua, zt = rs.standard_normal((B, N, 3)), rs.uniform(size=(B, N)), rs.standard_normal((B, N, 3))
    for b, n in enumerate(lens):
        q = rs.standard_normal((n, 4)); q /= np.linalg.norm(q, axis=-1, keepdims=True)
        r0[b, :n, :4] = q; r0[b, :n, 4:] = rs.standard_normal((n, 3)) * 8; mask[b, :n] = 1
    out = eng.forward_marginal_batch(torch.tensor(r0), ts, za, ua, zt, mask)
    for b, n in enumerate(lens):
        one = eng.forward_marginal(torch.tensor(r0[b, :n]), ts[b], za[b, :n], ua[b, :n], zt[b, :n])
        for k in ("rigids_t", "rot_score", "trans_score"):
            assert np.array_equal(out[k][b, :n].cpu().numpy(), one[k].cpu().numpy()), (b, k)          # same kernel: bit-exact
            assert float(out[k][b, n:].abs().sum()) == 0.0, (b, k)                                     # zero padding
        assert out["rot_score_scaling"][b] == one["rot_score_scaling"] and out["trans_score_scaling"][b] == one["trans_score_scaling"]
    # against the oracle (numpy RNG feeding both): example 0
    np.random.seed(3)
    n = lens[0]
    z1, u1 = np.random.randn(n, 3), np.random.rand(n)
    np.random.seed(3)
    ref = fo.forward_marginal(torch.tensor(r0[0, :n]).double(), ts[0])
    # the oracle draws the translation noise as normal(loc, scale): reproduce the standard normal it consumed
    np.random.seed(3); np.random.randn(n, 3); np.random.rand(n); z3 = np.random.normal(size=(n, 3))
    o1 = eng.forward_marginal_batch(torch.tensor(r0[:1]), ts[:1], z1[None].repeat(1, 0) if False else np.pad(z1, ((0, N - n), (0, 0)))[None],
                                    np.pad(u1, (0, N - n))[None], np.pad(z3, ((0, N - n), (0, 0)))[None], mask[:1])
    assert_close(o1["rot_score"][0, :n].cpu().numpy(), ref["rot_score"], 0, norm_rel=1e-6, name="rot_score vs oracle")
    assert_close(fo.quat_to_rotmat(o1["rigids_t"][0, :n, :4].cpu()).numpy(), fo.quat_to_rotmat(torch.as_tensor(ref["rigids_t"])[..., :4].float()).numpy(), 0,
                 atol=5e-6, name="rot_t vs oracle")


def test_ca_metrics_vs_oracle_and_reference_golden(eng):
    g = golden("metrics")
    N = 128
    ca = np.zeros((3, N, 3), np.float32); nv = []
    for k in range(3):
        x = g[f"ca_{k}"]; ca[k, :len(x)] = x; nv.append(len(x))
    m = eng.ca_metrics(torch.tensor(ca), nv)
    got = np.stack([m[k].cpu().numpy() for k in ("ca_ca_bond_dev", "ca_ca_valid_percent", "num_ca_steric_clashes", "ca_steric_clash_percent")], -1)
    for k in range(3):
        assert_close(got[k], g[f"ref_{k}"], 1e-6, atol=1e-9, name=f"metrics {k} vs the reference functions")
        dev, valid = fo.ca_ca_distance(ca[k, :nv[k]]); ncl, pcl = fo.ca_ca_clashes(ca[k, :nv[k]])
        assert_close(got[k], np.array([dev, valid, ncl, pcl], dtype=np.float64), 1e-6, atol=1e-9, name=f"metrics {k} vs oracle")
        assert got[k][2] == g[f"ref_{k}"][2]                                                          # clash COUNT: integer, bit-exact


def test_forward_use_cached_score_lookup(eng):
    """SO3Diffuser.use_cached_score=True (so3_diffuser.py:291-298): the head's bucketize + gather from the precomputed score-norm rows vs
    the oracle's restatement of that branch.  The look-up is a step function of the angle, so an angle within rounding of a grid point may
    land in the neighbouring bucket: all but a handful of residues must agree to 1e-6, the rest to the neighbouring table entry."""
    np.random.seed(31)
    B, N = 2, 80
    r7 = torch.stack([fo.sample_ref(N) for _ in range(B)])
    f = fo.init_feats(r7)
    f["t"] = torch.tensor([0.77, 0.36], dtype=torch.float64)
    with torch.no_grad():
        ref = fo.score_network_forward(fo.as_torch_weights(fo.synthetic_weights(0)), f, use_cached_score=True)
    eng.use_cached_score = True
    try:
        out = eng.forward(f)
        with pytest.raises(ValueError):
            eng.sample(1, 16, num_t=3)
    finally:
        eng.use_cached_score = False
    a, b = out["rot_score"].cpu().numpy(), ref["rot_score"].numpy()
    rel = np.abs(a - b).max(-1) / np.maximum(np.abs(b).max(-1), 1e-30)
    assert (rel < 1e-4).mean() > 0.97, f"only {(rel < 1e-4).mean():.3f} of the residues agree"
    assert rel.max() < 0.2                      # a neighbouring bucket, not garbage
    assert_close(out["trans_score"].cpu().numpy(), ref["trans_score"].numpy(), 0, norm_rel=1e-4, name="trans_score")


def test_sample_sharded_single_process_equals_sample_device(eng):
    """parallel.sample_sharded on the real engine (world size 1: no process group): same samples as the direct device loop, and a
    sub-range of the batch reproduces the corresponding samples of the full batch (the property the multi-GPU split relies on)."""
    from se3_diffusion_b200.parallel import sample_sharded, shard_range
    a37, rig, ms, nl = sample_sharded(eng, 4, 40, num_t=5, seed=21)
    b37, brig, _, _ = eng.sample_device(4, 40, num_t=5, seed=21, first_sample=0)
    assert torch.equal(a37, b37) and torch.equal(rig, brig)
    first, count = shard_range(4, 2, 1)
    c37, _, _, _ = eng.sample_device(count, 40, num_t=5, seed=21, first_sample=first)
    assert_close(c37.cpu().numpy(), a37[first:first + count].cpu().numpy(), 0, norm_rel=1e-5, name="rank-1 shard of a 2-way split")


@pytest.mark.parametrize("mode", ["sample", "train"])
def test_bench_dump_outputs(tmp_path, mode):
    """`bench.py --dump-outputs DIR` writes the last timed step's results as float .npy files; two runs with the same arguments use
    the same inputs, so they agree (sampling: both legs of a step compute the same samples)."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    extra = ["--num-t", "4", "--batch", "2"] if mode == "sample" else ["--batch", "1"]
    runs = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--mode", mode,
                            "--nres", "40", "--no-cpu-baseline", "--dump-outputs", str(d)] + extra,
                           cwd=tmp_path, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
        assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 2
        runs.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = runs
    assert all(v.dtype in (np.float32, np.float64) and np.all(np.isfinite(v)) for v in a.values())
    if mode == "sample":
        assert sorted(a) == ["atom37", "e2e_atom37", "e2e_psi", "e2e_rigids", "rigids"]
        assert a["atom37"].shape == (2, 40, 37, 3) and a["rigids"].shape == (2, 40, 7) and a["e2e_psi"].shape == (2, 40, 2)
        assert_close(a["e2e_atom37"], a["atom37"], 0, norm_rel=1e-5, name="host-buffer leg vs device leg")
        assert_close(a["e2e_rigids"][..., 4:], a["rigids"][..., 4:], 0, norm_rel=1e-5, name="host-buffer leg vs device leg")
        for k in a:
            assert_close(b[k], a[k], 0, norm_rel=1e-4, name=f"run 2 vs run 1: {k}")
        return
    assert sorted(a) == ["grads", "loss", "param_index", "params"]
    assert a["params"].shape == a["grads"].shape == a["param_index"].shape == (2_000_000,) and np.all(np.diff(a["param_index"]) > 0)
    assert np.array_equal(a["param_index"], b["param_index"])
    # the backward's atomic sums differ in rounding from run to run, and Adam turns rounding noise in a near-zero gradient into a step
    # of about lr: the runs agree to the tensor-core training mode's gradient accuracy, the parameters to 2 lr per Adam step
    adam_steps = 1 + 2 * 2                      # the warm-up step, then both legs of each timed step
    assert_close(b["params"], a["params"], 0, atol=2 * adam_steps * 1e-4, name="run 2 vs run 1: params")
    assert_close(b["grads"], a["grads"], 0, norm_rel=6e-3, name="run 2 vs run 1: grads")
    assert_close(b["loss"], a["loss"], 1e-3, name="run 2 vs run 1: loss")
