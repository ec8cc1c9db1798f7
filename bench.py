#!/usr/bin/env python
"""bench.py — sampled backbone residues/sec (N=256, 500 denoise steps) on N GPUs of one node.

  python bench.py --gpus 1 --steps K --warmup W            (our arm, default)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W            (one rank per GPU, NCCL)
  python bench.py --impl reference ...                     (the reference's CPU path = oracle port, host cores)

A "step" is one pass of the hot path over one batch: the whole reverse-diffusion sampling of B backbones per GPU
(prior draw -> 1 self-conditioning forward + (num_t-1) x [ScoreNetwork.forward + SE3Diffuser.reverse] + final forward ->
atom37), i.e. Experiment.inference_fn (experiments/train_se3_diffusion.py:718-818 of the reference) for that batch.
value = backbones x residues / step time, whole job (all GPUs).  Weak scaling: per-GPU batch fixed.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sampled backbone residues/sec (N=256, 500 denoise steps)"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--batch", type=int, default=None, help="backbones per GPU (default: 32 = BASELINE config 3's per-GPU shard)")
    p.add_argument("--nres", type=int, default=256)
    p.add_argument("--num-t", type=int, default=500)
    p.add_argument("--precision", default=None, choices=[None, "fp32", "bf16x3", "bf16"])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-steps", type=int, default=None, help="denoise steps of the bounded CPU sample")
    p.add_argument("--mode", default="sample", choices=["sample", "train"],
                   help="sample (default, the headline metric) | train: one optimiser step (fwd + DSM loss + bwd + all-reduce + Adam), BASELINE config 4")
    p.add_argument("--sweep", action="store_true", help="measure the other BASELINE configs (C1 paper weights, C2, C5 length sweep) in one run")
    p.add_argument("--lr", type=float, default=1e-4)
    p.add_argument("--train-gemm", default="tc", choices=["fp32", "bf16x3", "tc"],
                   help="training-path GEMMs: CUDA-core fp32 | split-bf16 mma.sync | split-bf16 with the edge-tensor GEMMs (forward, data and weight gradients) on tcgen05")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB in all) "
                        "so that two builds can be compared output for output")
    args = p.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.sweep):
        p.error("--dump-outputs applies to the GPU sampling and training runs (not --impl reference or --sweep)")
    return args


DUMP_LIMIT = 64 << 20


def write_dump(path, arrays):
    """Writes {name: float32 / float64 array} as path/<name>.npy."""
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT and all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), v)
    print(f"[bench] wrote {', '.join(sorted(arrays))} to {path}", file=sys.stderr)


def sample_subset(arrays):
    """Arrays indexed by global sample on axis 0: all of them if they fit DUMP_LIMIT, else the same fixed seeded subset of samples of
    each, whose indices go to sample_index."""
    n = next(iter(arrays.values())).shape[0]
    per_sample = sum(a.nbytes for a in arrays.values()) / n + 8
    if per_sample * n <= DUMP_LIMIT:
        return arrays
    keep = np.sort(np.random.default_rng(0).choice(n, int(DUMP_LIMIT // per_sample), replace=False))
    return dict({k: v[keep] for k, v in arrays.items()}, sample_index=keep.astype(np.float64))


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_baseline(nres, num_t, cpu_steps, state):
    """Bounded sample of the same workload on the host cores through the oracle port (kind "port"): 1 backbone x nres,
    the priming forward + `cpu_steps` denoise steps, extrapolated to the 501 forwards of a num_t-step sample."""
    import torch
    from oracle import framediff_oracle as fo
    w = fo.as_torch_weights(state)
    # thread count: the reference would use torch's default (all cores); on many-core hosts the elementwise-heavy IPA
    # temporaries scale badly, so calibrate on one small forward and keep the fastest setting (favours the baseline)
    ncpu = os.cpu_count() or 1
    cand = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    np.random.seed(7)
    fcal = fo.init_feats(fo.sample_ref(96)[None]); fcal["t"] = torch.ones(1)
    best, cores = None, cand[0]
    for c in cand:
        torch.set_num_threads(c)
        with torch.no_grad():
            fo.score_network_forward(w, fcal)
            t0 = time.perf_counter(); fo.score_network_forward(w, fcal); dtc = time.perf_counter() - t0
        if best is None or dtc < best:
            best, cores = dtc, c
    torch.set_num_threads(cores)
    np.random.seed(123)
    fo.igso3_row(fo.so3_t_to_idx(1.0))        # warm the IGSO(3) row cache (the reference's 52 s cache build is excluded too)
    r7 = fo.sample_ref(nres)[None]
    feats = fo.init_feats(r7)
    t0 = time.perf_counter()
    fo.inference_loop(w, feats, num_t=num_t, min_t=0.01, noise_scale=0.1, max_steps=cpu_steps)
    dt = time.perf_counter() - t0
    per_fwd = dt / (cpu_steps + 1)
    full = per_fwd * (num_t + 1)
    return {"value": nres / full, "unit": "residues/s", "cores": cores, "kind": "port",
            "sample": f"1 backbone x N={nres}: self-conditioning forward + {cpu_steps} of {num_t} denoise steps in {dt:.2f} s "
                      f"({per_fwd:.3f} s per forward+reverse), extrapolated x{num_t + 1}",
            "seconds_measured": dt}


def synthetic_state():
    from se3_diffusion_b200.synthetic import synthetic_weights      # deterministic random init of the architecture
    return synthetic_weights(0)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; /root/reference does not exist on
    the GPU box), all host threads.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import framediff_oracle as fo      # this arm never touches the product package or its .so
    state = fo.synthetic_weights(0)
    if args.mode == "train":                       # the reference's training step on the host (autograd through the port + torch Adam)
        vals, last = [], None
        for i in range(args.warmup + args.steps):
            last = cpu_train_baseline(args.nres, state, steps=4)
            if i >= args.warmup:
                vals.append(last["value"])
        v = float(np.mean(vals)); cb = dict(last); cb["value"] = v
        print(json.dumps({"impl": "reference", "metric": TRAIN_METRIC, "value": v, "unit": "examples/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic (random-init weights; one noised example)", "config": {"workload": f"train step, 1 example x N={args.nres}, CPU"},
                          "cpu_baseline": cb, "e2e": {"value": v, "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    args.cpu_steps = max(args.cpu_steps or 10, 10)       # SURVEY §8(d): at least 10 denoise steps per bounded sample (~9 s of host work per bench step)
    times = []
    last = None
    for i in range(args.warmup + args.steps):
        last = cpu_baseline(args.nres, args.num_t, args.cpu_steps, state)
        if i >= args.warmup:
            times.append(last["value"])
    v = float(np.mean(times))
    cb = dict(last); cb["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "residues/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * args.nres / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (random-init weights of the FrameDiff architecture, not weights/paper_weights.pth: throughput-neutral; "
                    "Gaussian/IGSO(3) prior noise)",
            "config": {"workload": f"1 backbone x N={args.nres} x {args.num_t} denoise steps per step, CPU (bounded sample, extrapolated)",
                       "nres": args.nres, "num_t": args.num_t},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "residues/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


TRAIN_METRIC = "training examples/sec (fwd + DSM loss + bwd + gradient all-reduce + Adam, N=256)"


def train_flops(B, N):
    """Executed FLOPs of one training step: forward (separable EdgeTransition / lookup layer-0 algebra, fd_forward_flops executed) +
    backward = 2x forward (dgrad + wgrad of every GEMM); loss and Adam are O(N^2) / O(params) and ignored."""
    n2 = float(N) * N
    fwd = (2248960.0 - 3 * (688128.0 - 524288.0)) * n2 + 32421376.0 * N       # dense layer-0 edge embedder in training (no table lookup)
    return 3.0 * fwd * B


def cpu_train_baseline(N, state, steps=6):
    """The reference's training step on the host: autograd through the oracle port (forward + loss_fn + backward) + torch Adam, 1 example."""
    import torch
    from oracle import framediff_oracle as fo
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    w = {k: v.clone().requires_grad_(True) for k, v in fo.as_torch_weights(state).items()}
    opt = torch.optim.Adam(list(w.values()), lr=1e-4)
    np.random.seed(3)
    r0 = fo.sample_ref(N).numpy().astype(np.float64); r0[:, 4:] *= 0.35
    fm = fo.forward_marginal(torch.tensor(r0), 0.5)
    tors = np.random.randn(N, 7, 2); tors /= np.linalg.norm(tors, axis=-1, keepdims=True)
    batch = {"rigids_0": torch.tensor(r0)[None], "rigids_t": fm["rigids_t"][None].float(), "rot_score": torch.tensor(fm["rot_score"])[None],
             "trans_score": torch.tensor(fm["trans_score"])[None], "rot_score_scaling": torch.tensor([fm["rot_score_scaling"]]),
             "trans_score_scaling": torch.tensor([fm["trans_score_scaling"]]), "res_mask": torch.ones(1, N, dtype=torch.float64),
             "fixed_mask": torch.zeros(1, N, dtype=torch.float64), "seq_idx": torch.arange(1, N + 1)[None],
             "torsion_angles_sin_cos": torch.tensor(tors)[None], "sc_ca_t": torch.zeros(1, N, 3, dtype=torch.float64), "t": torch.tensor([0.5], dtype=torch.float64)}
    def one_step():
        out = fo.score_network_forward(w, batch, float_mask_quirk=True)
        loss = fo.loss_terms(out, batch)["total_loss"]
        opt.zero_grad(); loss.backward(); opt.step()

    one_step()                                       # untimed: first-touch allocations, thread pool start-up
    n, t0 = 0, time.perf_counter()
    while n < steps and (n == 0 or time.perf_counter() - t0 < 12.0):      # bounded sample: about 10 s of host work
        one_step(); n += 1
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "examples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} steps of 1 example x N={N}: forward + loss_fn + backward (torch autograd through the oracle port) + Adam in {dt:.2f} s "
                      f"(after one untimed step)",
            "seconds_measured": dt}


def run_train(args):
    """--mode train: BASELINE config 4 (B=8 examples/GPU x N=256, DDP over the ranks)."""
    import torch
    import torch.distributed as dist
    from se3_diffusion_b200 import FrameDiffEngine
    from se3_diffusion_b200.parallel import TrainStep
    from se3_diffusion_b200.synthetic import training_batch
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    B, N = args.batch or 8, args.nres
    eng = FrameDiffEngine(local, "fp32")
    eng.train_set_gemm(args.train_gemm)
    state = synthetic_state()
    ts = TrainStep(eng, state, lr=args.lr)
    ts.broadcast_parameters()
    batch = training_batch(eng, B, N, seed=1 + rank)
    FE = ("rigids_t", "res_mask", "fixed_mask", "seq_idx", "t", "sc_ca_t", "torsion_angles_sin_cos")
    dev_batch = {k: v.to(dev) for k, v in batch.items()}
    pin_batch = {k: v.pin_memory() for k, v in batch.items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def dev_step():
        return ts({k: dev_batch[k] for k in FE}, dev_batch)

    def e2e_step():
        hb = {k: v.to(dev, non_blocking=True) for k, v in pin_batch.items()}      # H2D of the whole batch from pinned memory
        loss = ts({k: hb[k] for k in FE}, hb)
        return float(loss.item())                                                  # D2H of the step's result

    for _ in range(args.warmup):
        dev_step()
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    dev_ms = e2e_ms = 0.0
    exposed = 0.0
    launches = 0
    losses = []
    for i in range(args.steps):          # the two legs interleaved step by step (same clock / power state)
        l0 = eng.launch_count()
        barrier(); ev[0].record(); dev_step(); ev[1].record(); barrier()
        dev_ms += ev[0].elapsed_time(ev[1]); exposed += ts.exposed_comm_ms(); launches += eng.launch_count() - l0
        barrier(); t0 = time.perf_counter(); losses.append(e2e_step()); barrier()
        e2e_ms += (time.perf_counter() - t0) * 1e3
    t = torch.tensor([dev_ms, e2e_ms, exposed], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s, e2e_s, exposed_ms = float(t[0]) / 1e3 / args.steps, float(t[1]) / 1e3 / args.steps, float(t[2]) / args.steps
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed step (the e2e leg of the last iteration): its loss, the parameters it updated in place and the gradients it
        # computed (identical on every rank after the all-reduce); 17.4 M floats each, so a fixed seeded sample of 2 M positions
        idx = np.sort(np.random.default_rng(0).choice(ts.params.numel(), 2_000_000, replace=False))
        at = torch.from_numpy(idx).to(dev)
        write_dump(args.dump_outputs, {"loss": np.array([losses[-1]], np.float64), "params": ts.params[at].cpu().numpy(),
                                       "grads": ts.grads[at].cpu().numpy(), "param_index": idx.astype(np.float64)})
    if rank == 0:
        pk = peaks()
        fl = train_flops(B, N)
        ach = fl / dev_s / 1e12
        h2d = int(sum(v.numel() * v.element_size() for v in batch.values()))
        cb = None if args.no_cpu_baseline else cpu_train_baseline(N, state)
        line = {"metric": TRAIN_METRIC, "value": world * B / dev_s, "unit": "examples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if args.train_gemm == "fp32" else "bf16x3 (split bf16 products, fp32 accumulate; fp32 activations, weights, gradients and Adam state)",
                "data": "synthetic (random-init weights; CA random-walk backbones noised with forward_marginal, SURVEY §8(d))",
                "config": {"workload": f"train step, {B} examples/GPU x N={N} (BASELINE config 4 per-GPU shard), DDP over {world} GPU(s)",
                           "batch_per_gpu": B, "global_batch": world * B, "nres": N, "parallelism": f"dp{world}", "optimizer": "Adam",
                           "l2": "not flushed: every layer streams the %.0f MB fp32 edge tensor (> 126 MB L2)" % (B * N * N * 128 * 4 / 1e6)},
                "e2e": {"value": world * B / e2e_s, "unit": "examples/s", "ms_per_step": e2e_s * 1e3, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8},
                "comm_exposed_ms_per_step": exposed_ms, "allreduce_bytes_per_step": int(ts.grads.numel() * 4) if world > 1 else 0,
                "final_loss": losses[-1] if losses else None, "clocks": clk, "gpu_launches": int(launches),
                "roofline": {"bound": "tensor", "kernel": "whole training step (forward + dgrad + wgrad GEMMs: %s)" % {"fp32": "fp32 CUDA cores", "bf16x3": "mm3_kernel, mma.sync split-bf16", "tc": "edge-tensor forward / dgrad / wgrad on tc_gemm_kernel (tcgen05), node path and small weight gradients on mm3_kernel (mma.sync); split-bf16"}[args.train_gemm],
                             "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"],
                             "peak_source": pk["source"], "traffic": None, "executed_flops_per_step": fl},
                "cpu_baseline": cb}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def sample_line(args, eng, state, B, N, T, prec, world, rank, local, dist, torch, steps, warmup, tag, with_roofline=True, with_cpu=True, warm_T=None):
    """One sampling measurement (value + e2e legs interleaved step by step) -> the JSON line dict (rank 0) or None."""
    dev = torch.device("cuda", local)
    first = rank * B

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    gathered = torch.empty(world * B, N, 37, 3, device=dev) if world > 1 else None
    last = {}

    def device_step(seed, num_t=T):
        """inputs resident in HBM: prior drawn on the device, final coordinates stay in HBM (+ NCCL gather for N>1)."""
        a37, rig, ms, nl = eng.sample_device(B, N, num_t=num_t, seed=seed, first_sample=first)
        if world > 1:
            dist.all_gather_into_tensor(gathered, a37)
        last["a37"] = gathered if world > 1 else a37
        last["rig"] = rig
        return ms, nl

    masks = {"res_mask": np.ones((B, N), np.float32), "fixed_mask": np.zeros((B, N), np.float32),
             "seq_idx": np.tile(np.arange(1, N + 1, dtype=np.int32), (B, 1))}

    def e2e_step(seed):
        """public API with HOST buffers: init features H2D, final atom37/rigids/psi D2H into pinned memory."""
        return eng.sample(B, N, num_t=T, seed=seed, first_sample=first, **masks)

    for i in range(warmup):
        device_step(1000 + i, warm_T or T)
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    dev_wall = e2e_wall = gpu_ms = 0.0
    launches = 0
    for i in range(steps):                    # the two legs interleaved: same clock / power state for both
        barrier(); t0 = time.perf_counter()
        ms, nl = device_step(2000 + i)
        barrier(); dev_wall += time.perf_counter() - t0
        gpu_ms += ms; launches += nl
        barrier(); t0 = time.perf_counter()
        res = e2e_step(2000 + i)
        barrier(); e2e_wall += time.perf_counter() - t0
        if i == steps - 1:          # earlier steps' pinned output buffers go back to the allocator before the next step, as without a dump
            last["e2e"] = res
        del res
    # the loop runs on the engine's own stream and is timed there with CUDA events (fd_sample_dev's gpu_ms); wall adds the host-side
    # launch overhead and, for N>1, the NCCL gather — report the larger (honest) one, max over ranks
    t = torch.tensor([max(dev_wall, gpu_ms / 1e3), e2e_wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_s, e2e_s = float(t[0]) / steps, float(t[1]) / steps
    clk = clocks.stop() if rank == 0 else None
    # checksum of global samples 0..min(32, B)-1 of the LAST timed step (seed 2000+steps-1): Philox keys are (seed, global sample id), so
    # this number must be identical at 1, 2, 4 and 8 GPUs (SURVEY §8(e))
    nchk = min(32, B)
    chk = last["a37"][:nchk].double().sum().item() if rank == 0 else None
    chk_abs = last["a37"][:nchk].double().abs().sum().item() if rank == 0 else None
    if args.dump_outputs:
        # the last timed step's results of both legs (device-resident loop; public API with host buffers), in global-sample order
        e2e = last["e2e"]
        out = {"atom37": last["a37"], "rigids": last["rig"], "e2e_atom37": torch.from_numpy(e2e["prot_traj"][0]).to(dev),
               "e2e_rigids": torch.from_numpy(e2e["rigids_final"]).to(dev), "e2e_psi": torch.from_numpy(e2e["psi_pred"][0]).to(dev)}
        if world > 1:          # after the timed region: the timed path gathers atom37 only
            for k in ("rigids", "e2e_atom37", "e2e_rigids", "e2e_psi"):
                g = out[k].new_empty((world * B,) + tuple(out[k].shape[1:]))
                dist.all_gather_into_tensor(g, out[k].contiguous())
                out[k] = g
        if rank == 0:
            write_dump(args.dump_outputs, sample_subset({k: v.cpu().numpy() for k, v in out.items()}))
    if rank != 0:
        return None
    roof = None
    if with_roofline:
        from se3_diffusion_b200.synthetic import init_feats, random_frames
        pk = peaks()
        f = init_feats(random_frames(B, N, seed=0), t=0.5)
        eng.forward(f, want_atoms=False); torch.cuda.synchronize(dev)
        eng.stage_timing(True)
        reps = 3
        for _ in range(reps):
            eng.forward(f, want_atoms=False)
        torch.cuda.synchronize(dev)
        st = eng.stage_times()
        eng.stage_timing(False)
        et_ms = st["edge_transition"][0] / reps / 3            # per EdgeTransition layer (3 per forward)
        flops_layer = 524288.0 * B * N * N                     # executed FLOP/edge: 2*(128*384 + 384*384 + 512*128)
        ach = flops_layer / (et_ms * 1e-3) / 1e12
        fwd_ms = sum(v[0] for v in st.values()) / reps
        passes = 3 if prec == "bf16x3" else 1
        # dram__bytes_read+write of the kernel from one `ncu --set full` capture, regenerated by tools/ncu_traffic.sh; only used while the
        # capture was taken from THIS library version (fd_version) and precision — otherwise null rather than a stale constant
        traffic, tsrc = None, None
        for name in sorted(os.listdir(os.path.join(ROOT, "profiles")), reverse=True):
            if name.endswith("_fused_dram_traffic.json"):
                tj = json.load(open(os.path.join(ROOT, "profiles", name)))
                if tj.get("precision") == prec and tj.get("lib_version") == eng.lib.fd_version().decode():
                    traffic, tsrc = tj["dram_bytes_per_edge"] * B * N * N, name
                break
        roof = {"bound": "tensor", "kernel": "tc_edge_fused_kernel (EdgeTransition: 3 chained GEMMs + LayerNorm, one launch per layer; stage also holds "
                                             "the two O(N) node-term linears)",
                "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops_sustained"],
                "peak_source": pk["source"] + ", sustained bf16 figure (kernel timed inside a long step)",
                "mma_passes": passes, "mma_issue_tflops": ach * passes, "mma_issue_frac_of_peak": ach * passes / pk["bf16_tflops_sustained"],
                "note": "achieved = ALGORITHMIC FLOPs (524,288 per edge, DESIGN.md §4) / event time; in bf16x3 every product is three bf16 MMAs",
                "traffic": traffic, "traffic_source": tsrc, "algorithmic_bytes_per_launch": (1024 if prec == "bf16x3" else 512) * B * N * N,
                "ms_per_launch_group": et_ms, "algorithmic_flops_per_launch_group": flops_layer,
                "share_of_forward": st["edge_transition"][0] / reps / fwd_ms,
                "stage_ms_per_forward": {k: v[0] / reps for k, v in st.items()},
                "end_to_end": {"reference_equivalent_flops_per_residue": (2248960.0 * N * N + 32421376.0 * N) * (T + 1) / N,
                               "achieved_tflops_reference_equivalent": (2248960.0 * N * N + 32421376.0 * N) * (T + 1) * B / step_s / 1e12,
                               "frac_of_sustained_bf16_peak": (2248960.0 * N * N + 32421376.0 * N) * (T + 1) * B / step_s / 1e12 / pk["bf16_tflops_sustained"]}}
    value = world * B * N / step_s
    e2e_v = world * B * N / e2e_s
    cb = cpu_baseline(N, T, args.cpu_steps or 14, state) if with_cpu else None       # ~11 s of host work
    return {"metric": METRIC if (N == 256 and T == 500) else f"sampled backbone residues/sec (N={N}, {T} denoise steps)", "value": value,
            "unit": "residues/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (split bf16, fp32 accumulate)", "bf16": "bf16"}[prec],
            "data": "synthetic (random-init weights of the FrameDiff architecture; Philox Gaussian/IGSO(3) prior + step noise)" if tag != "C1"
                    else "weights/paper_weights.npz (the reference's shipped checkpoint); Philox prior + step noise",
            "config": {"workload": f"{B} backbones/GPU x N={N} residues x {T} denoise steps ({tag})",
                       "batch_per_gpu": B, "global_batch": world * B, "nres": N, "num_t": T, "precision": prec,
                       "parallelism": f"batch-sharded dp{world}", "cuda_graph": True,
                       "l2": "not flushed: each forward streams a %.0f MB edge tensor (> 126 MB L2)" % (B * N * N * 128 * 4 / 1e6)},
            "e2e": {"value": e2e_v, "unit": "residues/s", "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(sum(v.nbytes for v in masks.values())),
                    "d2h_bytes_per_step": int(B * N * (111 + 7 + 2) * 4)},
            "gpu_launches": int(launches), "gpu_ms_per_step_events": gpu_ms / steps,
            "sample_checksum": {"samples": nchk, "seed": 2000 + steps - 1, "sum": chk, "abs_sum": chk_abs},
            "clocks": clk, "roofline": roof, "cpu_baseline": cb}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.mode == "train":
        return run_train(args)
    import torch
    import torch.distributed as dist
    from se3_diffusion_b200 import FrameDiffEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if world != args.gpus and rank == 0:
        print(f"[bench] warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    torch.cuda.set_device(local)
    prec = args.precision or os.environ.get("FD_PRECISION", "bf16x3")   # parity-grade tensor-core mode (1e-4 vs the fp32 reference)
    eng = FrameDiffEngine(local, prec)
    state = synthetic_state()
    eng.load_weights(state)
    if args.sweep:
        # the other BASELINE configs (builder-run; JSON kept under profiles/): C1 with the shipped checkpoint, C2, and the C5 length sweep
        lines = []
        wpath = os.path.join(ROOT, "weights", "paper_weights.npz")
        cfgs = [("C2: BASELINE config 2", 32, 128, 500, 2)] + [(f"C5: length sweep N={n}", 32, n, 500, 1) for n in (100, 200, 300, 400, 512)]
        if os.path.exists(wpath):
            eng.load_weights(dict(np.load(wpath)))
            ln = sample_line(args, eng, state, 1, 60, 50, prec, world, rank, local, dist, torch, 5, 3, "C1", with_cpu=False)
            if ln: lines.append(ln)
            eng.load_weights(state)
        for tag, B, N, T, steps in cfgs:
            ln = sample_line(args, eng, state, B, N, T, prec, world, rank, local, dist, torch, steps, 3, tag, with_cpu=False, warm_T=10)
            if ln: lines.append(ln)
        if rank == 0:
            print(json.dumps({"sweep": lines}), flush=True)
    else:
        B = args.batch or 32
        line = sample_line(args, eng, state, B, args.nres, args.num_t, prec, world, rank, local, dist, torch, args.steps, args.warmup,
                           "BASELINE config 3 per-GPU shard" if (B == 32 and args.nres == 256) else "custom", with_cpu=not args.no_cpu_baseline)
        if rank == 0:
            print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
