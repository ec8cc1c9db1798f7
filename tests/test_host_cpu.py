"""CPU-side tests (-m "not gpu"): C-ABI surface, host logic, drop-in overlay, multi-process sharding logic (gloo)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import framediff_oracle as fo


def test_cabi_library_loads_and_exports_every_declared_symbol():
    from se3_diffusion_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "framediff_b200.h")).read()
    declared = set(re.findall(r"\b(fd_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 25
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/framediff_b200.h but not exported"
        assert name in _lib.SYMBOLS, f"{name} has no ctypes prototype in se3_diffusion_b200/_lib.py"
    assert lib.fd_version().decode().startswith("framediff_b200")


def test_param_schema_matches_reference_state_dict_layout():
    from se3_diffusion_b200.engine import param_schema
    ours = param_schema()
    assert ours == [(n, tuple(s)) for n, s in fo.param_schema()]
    assert len(ours) == 282 and sum(int(np.prod(s)) for _, s in ours) == 17446190   # SURVEY §6: 17,446,190 parameters


def test_forward_flops_model():
    from se3_diffusion_b200 import _lib
    lib = _lib.load()
    assert lib.fd_forward_flops(1, 256, 0) == 2248960 * 256 * 256 + 32421376 * 256   # SURVEY §8(d) F(N)
    assert lib.fd_forward_flops(3, 128, 1) < lib.fd_forward_flops(3, 128, 0)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    from se3_diffusion_b200 import FrameDiffEngine, FrameDiffError
    with pytest.raises(FrameDiffError):
        FrameDiffEngine(0)


def test_score_network_module_is_state_dict_compatible():
    from se3_diffusion_b200.score_network import ScoreNetwork
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_harness as rh
    mc, dc = rh.default_conf()
    net = ScoreNetwork(mc, diffuser=None)
    sd = net.state_dict()
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == [(n, tuple(s)) for n, s in fo.param_schema()]
    syn = {k: torch.tensor(v) for k, v in fo.synthetic_weights(0).items()}
    net.load_state_dict(syn, strict=True)
    net.load_state_dict({"module." + k: v for k, v in syn.items()}, strict=False)   # DataParallel-style keys are simply ignored
    with pytest.raises(RuntimeError):
        net.eval()
        with torch.no_grad():
            net({"rigids_t": torch.zeros(1, 4, 7)})        # CPU tensors: loud failure, no fallback
    bad = rh.to_attr({**mc, "ipa": {**mc.ipa, "no_heads": 4}})
    with pytest.raises(ValueError):
        ScoreNetwork(bad, None)


@pytest.mark.skipif(not os.path.isdir("/root/reference/model"), reason="reference tree not present (GPU box)")
def test_overlay_drop_in_with_reference_tree():
    """PEP-420 overlay: our model.score_network / data.se3_diffuser shadow the reference's, everything else still resolves to
    the reference; both shipped checkpoints load strict=True; the reference loads a state_dict written by our module."""
    code = r'''
import sys
sys.path.insert(0, "%(root)s/tests/golden"); sys.path.insert(0, "%(root)s")
import ref_harness as rh
rh.install_stubs()
sys.path.insert(0, "%(root)s/se3_diffusion_b200/overlay")
from model import score_network, ipa_pytorch
from data import se3_diffuser, all_atom
assert "se3_diffusion_b200/overlay" in score_network.__file__ and "se3_diffusion_b200/overlay" in se3_diffuser.__file__
assert ipa_pytorch.__file__.startswith("/root/reference") and all_atom.__file__.startswith("/root/reference")
mc, dc = rh.default_conf()
net = score_network.ScoreNetwork(mc, se3_diffuser.SE3Diffuser(dc))
for name in ("paper_weights.pth", "best_weights.pth"):
    net.load_state_dict(rh.load_reference_checkpoint(name), strict=True)
ref_net, _ = rh.build_reference(net.state_dict())
# analysis.utils: the overlay module re-exports the reference's and swaps only the PDB writer
from analysis import utils as au, metrics
import se3_diffusion_b200.pdb_writer as pw
assert "se3_diffusion_b200/overlay" in au.__file__ and metrics.__file__.startswith("/root/reference")
assert au.write_prot_to_pdb is pw.write_prot_to_pdb and callable(au.create_full_prot) and au.CA_IDX == 1
print("OVERLAY-OK", len(net.state_dict()))
''' % {"root": ROOT}
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert "OVERLAY-OK 282" in out.stdout, out.stdout + out.stderr


def test_state_dict_layout_equals_the_reference_module_and_shipped_checkpoints():
    """Our module's state_dict has exactly the parameter names, order and shapes of the reference's ScoreNetwork and of both shipped
    checkpoints (tests/golden/make_golden_overlay.py): the checkpoints load strict=True and the reference loads what our module writes."""
    from conftest import golden
    from se3_diffusion_b200.score_network import ScoreNetwork
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import ref_harness as rh
    g = golden("state_dict_layout")
    net = ScoreNetwork(rh.default_conf()[0], diffuser=None)
    ours = [(k, tuple(v.shape)) for k, v in net.state_dict().items()]
    for tag in ("module", "paper_weights", "best_weights"):
        dims = iter(g[f"{tag}_dims"].tolist())
        ref = [(str(n), tuple(next(dims) for _ in range(k))) for n, k in zip(g[f"{tag}_names"], g[f"{tag}_ndim"].tolist())]
        assert ours == ref, tag
        net.load_state_dict({n: torch.zeros(s) for n, s in ref}, strict=True)


def test_shard_range_partitions_batch():
    from se3_diffusion_b200.parallel import shard_range
    for B in (1, 7, 32, 256):
        for W in (1, 2, 3, 8):
            spans = [shard_range(B, W, r) for r in range(W)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == B
            for (f0, c0), (f1, _) in zip(spans, spans[1:]):
                assert f0 + c0 == f1
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1
    with pytest.raises(ValueError):
        shard_range(8, 2, 2)


_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
from se3_diffusion_b200.parallel import shard_range, gather_samples, sample_sharded
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%(port)d", rank=int(sys.argv[1]), world_size=2)
rank = dist.get_rank()
class FakeEngine:      # stands in for the CUDA engine: sample g's output depends only on its global index (Philox contract)
    def sample_device(self, B, N, first_sample=0, **kw):
        g = torch.arange(first_sample, first_sample + B, dtype=torch.float32)
        a37 = g[:, None, None, None].expand(B, N, 37, 3).clone()
        rig = g[:, None, None].expand(B, N, 7).clone() * 2
        return a37, rig, 1.0, 10
GB, N = 7, 5                                             # ragged: rank 0 owns 4 samples, rank 1 owns 3
a37, rig, ms, nl = sample_sharded(FakeEngine(), GB, N)
assert a37.shape == (GB, N, 37, 3) and rig.shape == (GB, N, 7)
assert torch.equal(a37[:, 0, 0, 0], torch.arange(GB, dtype=torch.float32)), a37[:, 0, 0, 0]
assert torch.equal(rig[:, 0, 0], 2 * torch.arange(GB, dtype=torch.float32))
t = torch.tensor([float(rank + 1)]); dist.all_reduce(t, op=dist.ReduceOp.MAX); assert t.item() == 2.0   # max-over-ranks timing reduction
dist.barrier(); dist.destroy_process_group()
print("RANK-OK", rank)
'''


def test_sharded_sampling_host_logic_gloo_world2(tmp_path):
    port = 29500 + (os.getpid() % 500)
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT, "port": port})
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"RANK-OK {r}" in o, o


def test_package_synthetic_weights_equal_the_oracles():
    """bench.py / tools generate weights with se3_diffusion_b200.synthetic (product side, never imports oracle/); they are the very
    arrays the parity tests use from the oracle (same schema order, same MT19937 stream)."""
    from oracle import framediff_oracle as fo
    from se3_diffusion_b200 import synthetic
    a, b = synthetic.synthetic_weights(0), fo.synthetic_weights(0)
    assert list(a) == list(b) and len(a) == 282
    assert all(np.array_equal(a[k], b[k]) for k in a)
    f = synthetic.init_feats(synthetic.random_frames(2, 16, seed=1))
    assert f["rigids_t"].shape == (2, 16, 7) and torch.allclose(f["rigids_t"][..., :4].norm(dim=-1), torch.ones(2, 16), atol=1e-6)


def test_product_code_never_imports_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline / reference legs may touch oracle/."""
    import re
    offenders = []
    for root in ("se3_diffusion_b200", "tools"):
        for dp, _, fns in os.walk(os.path.join(ROOT, root)):
            for fn in fns:
                if fn.endswith(".py") and re.search(r"^\s*(from|import)\s+oracle\b", open(os.path.join(dp, fn)).read(), re.M):
                    offenders.append(os.path.join(dp, fn))
    assert not offenders, offenders
    src = open(os.path.join(ROOT, "bench.py")).read()
    legs = [m.start() for m in re.finditer(r"^\s*from oracle import", src, re.M)]
    allowed = [src.index("def cpu_baseline"), src.index("def run_reference")] if "def cpu_baseline" in src else []
    for pos in legs:        # every oracle import sits inside the CPU-baseline or the reference-arm function
        fn_start = max(m.start() for m in re.finditer(r"^def \w+", src[:pos], re.M))
        assert src[fn_start:fn_start + 40].startswith(("def cpu_baseline", "def cpu_train_baseline", "def run_reference")), src[fn_start:fn_start + 60]


def test_grad_buckets_partition_the_arena():
    """The four backward stages' gradient buckets are contiguous, disjoint, cover the whole flat arena and follow the order the stages
    finish in (block 3 + torsion head first, embedders + block 0 last)."""
    from se3_diffusion_b200.engine import arena_layout
    from se3_diffusion_b200.parallel import grad_buckets
    lay, total = arena_layout()
    bk = grad_buckets()
    assert len(bk) == 4 and bk[0][1] == total and bk[3][0] == 0
    assert all(bk[i][0] == bk[i + 1][1] for i in range(3)) and all(lo < hi for lo, hi in bk)
    where = {n: next(i for i, (lo, hi) in enumerate(bk) if lo <= off < hi) for n, _, off in lay}
    assert where["score_model.torsion_pred.linear_1.weight"] == 0 and where["score_model.trunk.ipa_3.linear_q.weight"] == 0
    assert where["score_model.trunk.edge_transition_2.trunk.0.weight"] == 1 and where["score_model.trunk.ipa_1.linear_q.weight"] == 2
    assert where["embedding_layer.edge_embedder.0.weight"] == 3 and where["score_model.trunk.bb_update_0.linear.weight"] == 3
    assert sum(int(np.prod(s)) for _, s, _ in lay) == 17446190          # SURVEY §8(e): 17,446,190 fp32 parameters


def test_train_step_allreduce_logic_gloo():
    """World-size-2 gloo run of TrainStep's communication logic with a fake engine (the CUDA path cannot run here): after the step each
    rank's gradient arena holds the SUM over ranks on every bucket, and the Adam scale is 1/world."""
    code = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, "%(root)s")
from se3_diffusion_b200 import parallel
rank = int(os.environ["RANK"])
dist.init_process_group("gloo", rank=rank, world_size=2)
class FakeEngine:
    device = torch.device("cpu")
    def train_bind(self, p, g): self.g = g
    def train_forward(self, feats): return {}
    def loss_forward(self, out, batch, conf): return {"total_loss": torch.tensor(float(rank))}
    def loss_backward(self, out, batch, conf): return {}
    def train_backward(self, dout, s0, s1):
        lo, hi = parallel.grad_buckets()[s0]
        self.g[lo:hi] += (rank + 1) * (s0 + 1)
    def adam_step(self, p, g, m, v, step, lr, betas, eps, grad_scale): self.scale = grad_scale; self.snapshot = g.clone()
import se3_diffusion_b200.engine as E
parallel_flat = E.flat_from_state
E.flat_from_state = lambda state, device: torch.zeros(E.arena_layout()[1])
eng = FakeEngine()
ts = parallel.TrainStep(eng, {}, lr=1e-3)
torch.cuda.Event = lambda **k: type("Ev", (), {"record": lambda s: None, "synchronize": lambda s: None, "elapsed_time": lambda s, o: 0.0})()
ts({}, {})
ok = eng.scale == 0.5
for s, (lo, hi) in enumerate(parallel.grad_buckets()):
    ok = ok and bool(torch.all(eng.snapshot[lo:hi] == 3.0 * (s + 1)))
print("DDP-LOGIC-OK" if ok else "DDP-LOGIC-BAD", rank)
dist.destroy_process_group()
''' % {"root": ROOT}
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=300) for p in procs]
    for r, (o, e) in enumerate(outs):
        assert f"DDP-LOGIC-OK {r}" in o, o + e


def test_linear_initialisers_follow_the_reference_distribution():
    """SURVEY row a8: `_Linear` inits (model/ipa_pytorch.py:101-166): 'default' = LeCun truncated normal (std^2 = 1/fan_in after the
    truncation correction), 'relu' = He (2/fan_in), 'final' = zeros, biases zero."""
    from se3_diffusion_b200.score_network import _Linear
    torch.manual_seed(0)
    for init, scale in (("default", 1.0), ("relu", 2.0)):
        lin = _Linear(512, 768, init)
        w = lin.weight.detach().numpy()
        assert abs(w.std() - np.sqrt(scale / 512)) < 0.02 * np.sqrt(scale / 512), (init, w.std())
        assert np.abs(w).max() <= 2.0 * np.sqrt(scale / 512) / 0.87962566103423978 + 1e-6      # truncated at +-2 sigma of the parent normal
        assert float(lin.bias.abs().max()) == 0.0
    lin = _Linear(64, 32, "final")
    assert float(lin.weight.abs().max()) == 0.0
    with pytest.raises(ValueError):
        _Linear(4, 4, "nonsense")


@pytest.mark.parametrize("mode", ["sample", "train"])
def test_bench_reference_arm_contract(mode):
    """`bench.py --impl reference` (the CPU arm the driver times next to the product): runs without the product library, prints ONE JSON line with
    the contract's keys, e2e repeating the line's own value, and a cpu_baseline block describing the bounded sample."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    # run in-process-of-the-child through runpy so the child can inspect its own address space afterwards: the product library must not be mapped
    prog = ("import runpy, sys; sys.argv = ['bench.py', '--impl', 'reference', '--mode', '%s', '--steps', '1', '--warmup', '0', '--nres', '24', "
            "'--num-t', '12']; runpy.run_path('bench.py', run_name='__main__'); "
            "assert 'libframediff' not in open('/proc/self/maps').read(), 'reference arm mapped the product library'" % mode)
    cmd = [sys.executable, "-c", prog]
    env = dict(os.environ, OMP_NUM_THREADS="8")
    res = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, res.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["higher_is_better"] is True and d["value"] > 0
    assert d["unit"] == ("residues/s" if mode == "sample" else "examples/s")
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    if mode == "sample":
        assert "10 of 12 denoise steps" in cb["sample"]          # at least 10 denoise steps per bounded sample (SURVEY §8(d))
