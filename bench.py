#!/usr/bin/env python
"""Benchmark of the separation hot path (driver contract: one JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]

Headline metric (BASELINE.json): Glow ``log_prob`` samples/s on synthetic mel-spectrogram patches of
the ``configs/melspec_glow.yml`` shape (96x64x1, L=3, K=40, 512 filters, learnable top prior),
random-init ("perturbed") weights.  One *step* = one ``log_prob`` pass over one batch of B patches per
GPU.  The second half of the metric, BASIS Langevin segment-steps/s with two Glow priors, is measured in
the same run and reported under ``"basis"``.

* ``value``  : whole-job samples/s, inputs resident in HBM, device time by CUDA events (per step, with
               an L2 flush between steps outside the events), max over ranks.
* ``e2e``    : the same metric through the public API (``Glow.log_prob`` -> C ABI) with the batch in
               PINNED HOST memory: H2D copy + compute + D2H of the [B] log-probabilities inside the
               timed region, every step.
* ``roofline``: the dominant kernel (k_nn_tc4, the fused tcgen05 coupling network): algorithmic conv
               FLOPs of the recorded launches / their summed CUDA-event time (events on the launching
               stream, recorded during the timed region) vs the measured sustained bf16 peak.
* ``cpu_baseline`` / ``--impl reference``: the reference-faithful CPU graph (oracle/glow_oracle.py,
               torch-CPU fp32, coupling network evaluated twice as the TFP graph does) on the host
               cores, on a bounded sample of the same workload.  TensorFlow 2.2 cannot be installed in
               this image, so kind = "port".

Multi-GPU (torchrun, one rank per GPU): the batch dimension shards with no data-path collective
("weak": B patches per GPU); NCCL is used only for the barrier and the max-over-ranks timing.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F_GLOW = 48.22e9          # FLOP per patch per coupling-network pass (BASELINE.md section 2)
D_PATCH = 96 * 64


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_sustained": float(p.get("bf16_tflops_sustained", 1378.1)), "bf16_burst": float(p.get("bf16_tflops", 1643.9)),
                "hbm": float(p.get("hbm_gbs", 6551.0)), "source": "measured"}
    return {"bf16_sustained": 1400.0, "bf16_burst": 1590.0, "hbm": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi SM clock / throttle reasons sampled every 200 ms while the timed region runs."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.strip().split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------ CPU reference arm
def _cpu_model(K: int):
    import torch
    from audiosourcesep_b200 import GlowConfig
    from audiosourcesep_b200.weights import init_glow_params
    from oracle.glow_oracle import GlowOracle
    cfg = GlowConfig(K=K)
    return cfg, GlowOracle(cfg, init_glow_params(cfg, seed=2), dtype=torch.float32)


def cpu_log_prob_rate(sample: int, K: int = 40, repeats: int = 1):
    """samples/s of the reference-faithful CPU graph on `sample` patches (all host threads)."""
    import torch
    from audiosourcesep_b200 import synthetic
    _, oracle = _cpu_model(K)
    x = torch.as_tensor(synthetic.mel_patches_db(sample, seed=0))
    best = None
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            oracle.log_prob_reference_graph(x)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return sample / best, best


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path.  The TF graph cannot run
    here (TensorFlow 2.2 / TFP 0.9 absent, no wheel, Python 3.12), so the reference-faithful port in
    oracle/ is timed with every host thread torch-CPU will use; rank 0 only."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 for its workers; the reference arm runs on rank 0 alone and takes every core
    try:
        torch.set_num_threads(max(torch.get_num_threads(), os.cpu_count() or 1))
    except RuntimeError:
        pass
    cores = torch.get_num_threads()
    sample = args.cpu_sample
    _, oracle = _cpu_model(args.K)
    from audiosourcesep_b200 import synthetic
    x = torch.as_tensor(synthetic.mel_patches_db(sample, seed=0))
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            lp = oracle.log_prob_reference_graph(x)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"log_prob": lp.numpy()})
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms * 1e-3)
    desc = (f"{sample} patches per step, reference-faithful graph (coupling network evaluated twice), torch-CPU fp32, "
            f"{cores} threads of {os.cpu_count()} logical cores")
    line = {
        "impl": "reference", "metric": "glow_log_prob_samples_per_s", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args, per_gpu_batch=sample, note="bounded CPU sample of the same workload"),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(directory, arrays, rank=0, world=1):
    """``--dump-outputs``: what the timed path returned in its last step, as ``<directory>/<name>.npy`` in float32
    (``<name>_rank<r>.npy`` per rank when several ranks run), so that two builds can be compared output for output."""
    os.makedirs(directory, exist_ok=True)
    suffix = "" if world == 1 else f"_rank{rank}"
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}{suffix}.npy"), np.ascontiguousarray(a, dtype=np.float32))


def _config(args, per_gpu_batch, note=None):
    c = {"workload": f"glow_log_prob melspec_glow.yml (96x64x1, L=3, K={args.K}, n_filters=512, learntop), "
                     f"{per_gpu_batch} patches per GPU per step",
         "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * args.gpus,
         "weights": "random-init (perturbed generator, seed 2)",
         "cache": "L2 flushed (512 MiB write) between timed steps, outside the CUDA-event brackets",
         "sharding": "patches sharded over ranks, no data-path collective"}
    if note:
        c["note"] = note
    return c


# ------------------------------------------------------------------------------------ our arm
# tcgen05 products per GEMM of every Glow precision mode: the roofline denominator of a mode is the measured sustained
# bf16 peak divided by this number (the extra products are the price of the mode, not useful work)
PRODUCTS = {"bf16": 1, "fp16": 1, "bf16x2": 2, "fp16x2": 2, "fp16x3": 3}


def _prec(_lib, name):
    return {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "fp16": _lib.PREC_FP16, "bf16x2": _lib.PREC_BF16X2,
            "fp16x2": _lib.PREC_FP16X2, "fp16x3": _lib.PREC_FP16X3}[name]


def parity_block(models_by_mode, torch, ops, bo, synthetic, D):
    """Gate values of every benchmarked Glow mode, measured in THIS run against the committed oracle vectors
    (tests/golden/glow_k40.npz: float64 oracle score / log_prob of the full-depth BASIS priors at n_mixed = 30, the
    inputs regenerated from the seeded generators; scores and states compared on the fixture's fixed half of the
    elements).  The oracle itself is not executed here."""
    path = os.path.join(ROOT, "tests", "golden", "glow_k40.npz")
    if not os.path.exists(path):
        return None
    gold = np.load(path)
    n = gold["logp1"].shape[0]
    keep = np.unpackbits(gold["keep"], count=n * D).reshape(n, 96, 64, 1).astype(bool)
    keep_d = torch.as_tensor(keep).cuda()
    oracle_score = {}
    for key in ("grad1", "grad2"):
        oracle_score[key] = np.zeros(keep.shape, np.float32)
        oracle_score[key][keep] = gold[key]
    mixed, _, _ = synthetic.basis_problem(n)
    x1, x2 = synthetic.langevin_init(n, seed=4)
    sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
    out = {"reference": "tests/golden/glow_k40.npz (float64 oracle, K=40, n_mixed=30, half of the score elements; "
                        "generator tests/golden/make_glow_k40_golden.py)",
           "gates": {"log_prob_nats_per_dim": 1e-3, "round_trip_max_abs": 1e-4, "langevin_step_state_rel": 1e-3}}
    for mode, (m1, m2) in models_by_mode.items():
        r = {}
        t1, t2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
        g1, lp1 = m1.grad_log_prob(t1, return_log_prob=True)
        g2, lp2 = m2.grad_log_prob(t2, return_log_prob=True)
        r["log_prob_err_nats_per_dim"] = float(max(np.max(np.abs(lp1.cpu().numpy() - gold["logp1"])),
                                                   np.max(np.abs(lp2.cpu().numpy() - gold["logp2"]))) / D)
        errs = []
        for g, key in ((g1, "grad1"), (g2, "grad2")):
            ref = gold[key].astype(np.float64)
            errs.append(float(np.linalg.norm(g.cpu().numpy()[keep] - ref) / np.linalg.norm(ref)))
        r["score_rel_l2_err"] = max(errs)
        z = m1.forward(t1)
        r["round_trip_max_abs"] = float((m1.inverse(z) - t1).abs().max().item())        # states are normalised units
        g_fn, gg_fn = None, None
        step = {}
        for idx in (0, 1, 2, 4, 9):
            eta, lam, ns = bo.langevin_step_constants(sig, idx)
            rng = np.random.Generator(np.random.PCG64(100 + idx))
            n1, n2 = (rng.standard_normal(x1.shape).astype(np.float32) for _ in range(2))
            # expected state: the fused update applied to the ORACLE scores (computed on the device by the same
            # Langevin kernel, whose own error is ~1e-7, tests/test_gpu_langevin.py); the update is element-wise, so it is
            # right wherever the oracle score is stored
            e1, e2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
            ops.langevin_step(e1, e2, torch.as_tensor(oracle_score["grad1"]), torch.as_tensor(oracle_score["grad2"]),
                              torch.as_tensor(mixed), float(eta), float(lam), float(ns), n1=torch.as_tensor(n1), n2=torch.as_tensor(n2))
            a1, a2 = torch.as_tensor(x1).cuda(), torch.as_tensor(x2).cuda()
            ops.basis_glow_inner(m1, m2, torch.as_tensor(mixed), a1, a2, 1, float(eta), float(lam), float(ns),
                                 noise1=torch.as_tensor(n1[None]), noise2=torch.as_tensor(n2[None]))
            step[f"sigma_idx_{idx}"] = float(max(torch.linalg.norm((a1 - e1)[keep_d]) / torch.linalg.norm(e1[keep_d]),
                                                 torch.linalg.norm((a2 - e2)[keep_d]) / torch.linalg.norm(e2[keep_d])).item())
        r["langevin_step_state_rel_err"] = step
        r["gates_met"] = {"log_prob": r["log_prob_err_nats_per_dim"] <= 1e-3, "round_trip": r["round_trip_max_abs"] <= 1e-4,
                          "langevin_step_at_sigma_idx": [i for i in (0, 1, 2, 4, 9) if step[f"sigma_idx_{i}"] <= 1e-3]}
        out[mode] = r
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: audiosourcesep_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from audiosourcesep_b200 import GlowConfig, _lib, ops, synthetic
    from audiosourcesep_b200.glow import Glow
    from audiosourcesep_b200.weights import init_glow_params
    # (the product path never touches oracle/: the sigma schedule and step constants come from the package)
    from audiosourcesep_b200.ncsn import utils as bo

    dev = torch.device("cuda", local_rank)
    peaks = _peaks()
    cfg = GlowConfig(K=args.K)
    params = init_glow_params(cfg, seed=2)
    model = Glow(cfg, params, precision=_lib.PREC_BF16, device=local_rank)
    B = args.batch

    def patches(n, seed):
        base = synthetic.mel_patches_db(min(n, 64), seed=seed)
        reps = (n + base.shape[0] - 1) // base.shape[0]
        # distinct patches: cyclic shifts of the seeded base set along time
        return np.ascontiguousarray(np.concatenate([np.roll(base, 3 * i, axis=2) for i in range(reps)], axis=0)[:n])

    x_host = torch.as_tensor(patches(B, 100 + rank)).pin_memory()
    x_dev = x_host.to(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(step_fn, steps, warmup, profile=False, do_flush=True, local=False):
        """local=True: a measurement only rank 0 makes (kernel-level profiles) -- no collective may be issued."""
        sync = torch.cuda.synchronize if local else barrier
        for _ in range(warmup):
            step_fn()
        sync()
        evs = []
        if profile == "conv":
            _lib.conv_profile(True)
        elif profile == "hbm":
            _lib.hbm_profile(True)
        elif profile:
            _lib.tc_profile(True)
        n0 = _lib.launch_count()
        for _ in range(steps):
            if do_flush:
                flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_fn()
            b.record()
            evs.append((a, b))
        sync()
        launches = _lib.launch_count() - n0
        prof = None
        if profile == "conv":
            prof = _lib.conv_profile_read()
            _lib.conv_profile(False)
        elif profile == "hbm":
            prof = {name: _lib.hbm_profile_read(cat) for name, cat in _lib.HBM_CATEGORIES.items()}
            _lib.hbm_profile(False)
        elif profile:
            prof = _lib.tc_profile_read()
            _lib.tc_profile(False)
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1 and not local:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, prof

    def tc_roofline(prof, total_ms, kernel, products):
        k_ms, k_launches, k_flops = prof
        achieved = k_flops / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
        peak = peaks["bf16_sustained"] / products
        return {"bound": "tensor", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "products_per_gemm": products,
                "peak_source": f"{peaks['source']} sustained bf16 ({peaks['bf16_sustained']:.1f} TFLOP/s; kernel timed inside a long step)"
                               + ("" if products == 1 else f" / {products} tcgen05 products per GEMM of this precision mode"),
                "launches": k_launches, "avg_launch_ms": k_ms / max(1, k_launches),
                "kernel_share_of_step": k_ms / total_ms if total_ms > 0 else None,
                "alg_flops_per_launch": k_flops / max(1, k_launches)}

    # ---- 1. device-resident throughput (value) with the kernel-level CUDA events for the roofline
    out = {}

    def step_dev():
        out["lp"] = model.log_prob(x_dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms, launches, prof = timed_loop(step_dev, args.steps, args.warmup, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms * 1e-3)
    lp = out["lp"].float().cpu().numpy()
    if not np.all(np.isfinite(lp)):
        raise SystemExit("non-finite log_prob in the benchmark batch")
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"log_prob": lp}, rank, world)
    roofline = tc_roofline(prof, total_ms, "k_nn_tc4<fwd> (fused conv3x3 -> conv1x1 -> conv3x3 coupling network, K-pipelined tcgen05)", 1)
    roofline["traffic"] = None

    # ---- 1b. the HBM-bound kernels of the same pass (fused flow step = ActNorm + 1x1 + coupling + log-det + col2im)
    nsub = max(2, args.steps // 2)
    hbm_ms, _, hprof = timed_loop(step_dev, nsub, 1, profile="hbm")
    roofline_hbm = []

    def hbm_entry(name, kernel, rec, note):
        ms, n, by = rec
        if n == 0 or ms <= 0:
            return
        gbs = by / (ms * 1e-3) / 1e9
        roofline_hbm.append({"bound": "hbm", "kernel": kernel, "category": name, "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                             "frac": gbs / peaks["hbm"], "launches": n, "avg_launch_us": 1e3 * ms / n,
                             "algorithmic_bytes_per_launch": by / n, "traffic": None, "note": note})

    hbm_entry("flow_step", "k_pre / k_post_pre<C, next, fused col2im>", hprof["flow_step"],
              f"log_prob at {B} patches: 12 C bytes per pixel per flow step (state in, network output, state out; SURVEY 8(d)); "
              "the fused col2im really reads the 9 per-tap fp32 partials of the tensor-core kernel instead of r")

    # ---- 2. end to end through the public API with host buffers
    def step_e2e():
        out["lp_host"] = model.log_prob(x_host.to(dev, non_blocking=True)).cpu()

    e2e_ms, _, _ = timed_loop(step_e2e, args.steps, args.warmup)
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)

    # ---- 2b. batch-size sweep of log_prob (config 1 at the reference's sizes: n_mixed = 30, training batch 32, ...)
    sweep = {}
    for n in [int(v) for v in args.sweep.split(",") if v]:
        xs = torch.as_tensor(patches(n, 200 + rank)).to(dev)
        nst = 5 if n <= 512 else 3
        s_ms, s_launches, _ = timed_loop(lambda: model.log_prob(xs), nst, 2)
        sweep[str(n)] = {"samples_per_s": world * n * nst / (s_ms * 1e-3), "ms_per_pass": s_ms / nst, "gpu_launches_per_pass": s_launches // nst,
                         "alg_tflops": world * n * nst * F_GLOW * (args.K / 40.0) / (s_ms * 1e-3) / 1e12}
        del xs

    # ---- 2c. the other directions of config 1 in every precision mode: inverse(z) and grad_log_prob(x), device-resident
    directions = {}
    for mode in [m for m in args.modes.split(",") if m]:
        if mode != "bf16":
            model.prepare(_prec(_lib, mode))
        prods = PRODUCTS[mode]
        d = {"products_per_gemm": prods}
        if mode != "bf16":
            l_ms, _, l_prof = timed_loop(step_dev, nsub, 1, profile=True)
            d["log_prob"] = {"value": world * B * nsub / (l_ms * 1e-3), "unit": "samples/s", "ms_per_step": l_ms / nsub,
                             "roofline": tc_roofline(l_prof, l_ms, "k_nn_tcx<fwd> (two-pass split-precision coupling network, tcgen05)", prods)}
        z_dev = model.forward(x_dev)

        def step_inv():
            out["xr"] = model.inverse(z_dev)

        inv_ms, inv_launches, _ = timed_loop(step_inv, nsub, 1)
        rt = float((out["xr"] - x_dev).abs().max().item()) / 120.0

        def step_grad():
            out["g"] = model.grad_log_prob(x_dev)

        g_ms, g_launches, _ = timed_loop(step_grad, nsub, 1)
        d["inverse"] = {"value": world * B * nsub / (inv_ms * 1e-3), "unit": "samples/s", "ms_per_step": inv_ms / nsub,
                        "gpu_launches": inv_launches, "alg_tflops": world * B * nsub * F_GLOW * (args.K / 40.0) / (inv_ms * 1e-3) / 1e12,
                        "round_trip_max_abs_normalised": rt, "gate": 1e-4, "gate_met": rt <= 1e-4}
        d["grad_log_prob"] = {"value": world * B * nsub / (g_ms * 1e-3), "unit": "samples/s", "ms_per_step": g_ms / nsub,
                              "gpu_launches": g_launches,
                              "alg_tflops": world * B * nsub * 2 * F_GLOW * (args.K / 40.0) / (g_ms * 1e-3) / 1e12}
        directions[mode] = d
        del z_dev
    del model

    # ---- 3. BASIS Langevin segment-steps/s with two Glow priors (second half of the metric), per precision mode, at the
    #         reference's n_mixed = 30 (run_basis_sep.py:478) and at a batch that fills the GPU
    basis, parity = None, None
    if args.basis_segments:
        bcfg = GlowConfig(K=args.K, minval=0.0, maxval=1.0)
        p1, p2 = init_glow_params(bcfg, seed=2), init_glow_params(bcfg, seed=3)
        sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
        eta, lam, ns = bo.langevin_step_constants(sig, 9)
        T = args.basis_T
        basis, pair_by_mode = {}, {}
        for mode in [m for m in args.basis_modes.split(",") if m]:
            m1 = Glow(bcfg, p1, precision=_prec(_lib, mode), device=local_rank)
            m2 = Glow(bcfg, p2, precision=_prec(_lib, mode), device=local_rank)
            pair_by_mode[mode] = (m1, m2)
            legs = {}
            for nseg in [int(v) for v in args.basis_segments.split(",") if v]:
                mixed, _, _ = synthetic.basis_problem(min(nseg, 32), seed1=10 + rank, seed2=50 + rank)
                mixed = np.concatenate([mixed] * ((nseg + mixed.shape[0] - 1) // mixed.shape[0]))[:nseg]
                x1, x2 = synthetic.langevin_init(nseg, seed=4 + rank)
                mixed_d = torch.as_tensor(mixed).to(dev)
                t1, t2 = torch.as_tensor(x1).to(dev), torch.as_tensor(x2).to(dev)
                stepno = [0]

                def step_basis():
                    ops.basis_glow_inner(m1, m2, mixed_d, t1, t2, T, float(eta), float(lam), float(ns), seed=1,
                                         step0=stepno[0], elem_offset=rank * nseg * D_PATCH)
                    stepno[0] += T

                nsteps = max(1, args.steps // 2)
                # 3 warm-up calls: eager pass + step-graph capture, capture of the N <= 128 score graphs, first pure replay
                b_ms, b_launches, _ = timed_loop(step_basis, nsteps, 3)
                legs[str(nseg)] = {"value": world * nseg * T * nsteps / (b_ms * 1e-3), "unit": "segment-steps/s", "segments_per_gpu": nseg,
                                   "ms_per_langevin_step": b_ms / (nsteps * T), "gpu_launches_per_langevin_step": b_launches // (nsteps * T),
                                   "alg_tflops": world * nseg * T * nsteps * 4 * F_GLOW * (args.K / 40.0) / (b_ms * 1e-3) / 1e12,
                                   "finite": bool(torch.isfinite(t1).all() and torch.isfinite(t2).all())}
            basis[mode] = {"metric": "basis_glow_segment_steps_per_s", "products_per_gemm": PRODUCTS[mode], "segments": legs,
                           "note": "2 priors x (forward + data-gradient) = 4 F_glow algorithmic FLOP per segment-step; in-kernel Philox "
                                   "noise; sigma index 9 of the 10-level schedule; the gate each mode meets is in `parity`"}
        if rank == 0 and args.parity:
            parity = parity_block(pair_by_mode, torch, ops, bo, synthetic, D_PATCH)
        # ---- the fused Langevin update alone at a size that spills L2 (HBM roofline of k_langevin)
        if rank == 0:
            nl = 4096
            shp = (nl, 96, 64, 1)
            g = torch.Generator(device=dev).manual_seed(0)
            ten = [torch.rand(shp, device=dev, generator=g) for _ in range(5)]

            def step_lan():
                ops.langevin_step(ten[0], ten[1], ten[2], ten[3], ten[4], 2e-5, 1e4, 6.3e-3, seed=1, step=0)

            _, _, lprof = timed_loop(step_lan, 5, 2, profile="hbm", do_flush=False, local=True)
            hbm_entry("langevin", "k_langevin<in-kernel Philox>", lprof["langevin"],
                      f"{nl} segments (7 tensors x 100 MB, larger than L2): 5 reads + 2 writes x 4 B per element (SURVEY 8(d))")
            del ten
        del pair_by_mode

    # ---- 4. BASIS with NCSN v1 / v2 score networks (configs 4 and 5 of BASELINE.json), n_mixed = 30 segments per GPU, in the
    #         throughput mode (one bf16 product) and the parity mode (three split-bf16 products)
    ncsn = {}
    if args.ncsn_segments > 0:
        from audiosourcesep_b200 import NCSNConfig
        from audiosourcesep_b200.ncsn.score_model import ScoreModel
        from audiosourcesep_b200.weights import init_ncsn_params
        nseg = args.ncsn_segments
        mixed, _, _ = synthetic.basis_problem(nseg, seed1=20 + rank, seed2=60 + rank)
        mixed_d = torch.as_tensor(mixed).to(dev)
        for ver, ncfg, gflop in (("v1", NCSNConfig(version="v1", ngf=192, num_classes=10, sigma1=1.0), 533.9),
                                 ("v2", NCSNConfig(version="v2", ngf=128, num_classes=200, sigma1=30.0), 237.3)):
            sig_n = bo.get_sigmas(ncfg.sigma1, ncfg.sigmaL, ncfg.num_classes, "logarithmic")
            for mode, prec, prods in (("bf16", _lib.PREC_BF16, 1), ("bf16x3", _lib.PREC_BF16X3, 3)):
                if mode not in args.ncsn_modes.split(","):
                    continue
                s1 = ScoreModel(ncfg, init_ncsn_params(ncfg, seed=11), sigmas=sig_n, device=local_rank, precision=prec)
                s2 = ScoreModel(ncfg, init_ncsn_params(ncfg, seed=12), sigmas=sig_n, device=local_rank, precision=prec)
                a1, a2 = synthetic.langevin_init(nseg, seed=7 + rank)
                u1, u2 = torch.as_tensor(a1).to(dev), torch.as_tensor(a2).to(dev)
                idx = ncfg.num_classes - 1
                eta_n, lam_n, ns_n = bo.langevin_step_constants(sig_n, idx)
                cnt = [0]

                def step_ncsn():
                    ops.basis_ncsn_inner(s1, s2, mixed_d, u1, u2, idx, args.ncsn_T, float(eta_n), float(lam_n), float(ns_n),
                                         seed=2, step0=cnt[0], elem_offset=rank * nseg * D_PATCH)
                    cnt[0] += args.ncsn_T

                nst = max(2, args.steps // 2)
                # rate: the shipped path (steps 2..T of a call replayed as one CUDA graph, the two networks as parallel
                # branches); kernel roofline / share: a second loop with per-launch events, which launches eagerly
                n_ms, n_launches, _ = timed_loop(step_ncsn, nst, 3)
                rate = world * nseg * args.ncsn_T * nst / (n_ms * 1e-3)
                p_ms, _, (c_ms, c_n, c_fl) = timed_loop(step_ncsn, 2, 0, profile="conv")
                # the x3 mode launches every convolution three times: its algorithmic FLOPs are those of ONE product
                conv_tf = c_fl / prods / (c_ms * 1e-3) / 1e12 if c_ms > 0 else 0.0
                peak = peaks["bf16_sustained"] / prods
                leg = {"metric": f"basis_ncsn_{ver}_segment_steps_per_s", "value": rate, "unit": "segment-steps/s",
                       "segments_per_gpu": nseg, "products_per_conv": prods, "ms_per_langevin_step": n_ms / (nst * args.ncsn_T),
                       "gpu_launches_per_langevin_step": n_launches // (nst * args.ncsn_T), "alg_tflops": rate * gflop / 1e3,
                       "roofline": {"bound": "tensor", "kernel": "k_conv_tc (TMA-fed tcgen05 implicit-GEMM convolution)",
                                    "achieved": conv_tf, "peak": peak, "unit": "TFLOP/s", "frac": conv_tf / peak, "launches": c_n,
                                    "kernel_share_of_step": c_ms / p_ms if p_ms > 0 else None,
                                    "profiled_loop": "eager launches with per-launch CUDA events (graph replay off), "
                                                     f"{p_ms / (2 * args.ncsn_T):.2f} ms per Langevin step",
                                    "peak_source": f"{peaks['source']} sustained bf16 / {prods} products per convolution"},
                       "step_roofline_frac": rate * gflop / 1e3 / world / peak,
                       "gate": ("per-step Langevin state <= 1e-3 at every noise level (tests/test_gpu_ncsn.py)" if prods == 3 else
                                "per-step gate met on the annealed end of the schedule only (score error 1-5 %)"),
                       "finite": bool(torch.isfinite(u1).all() and torch.isfinite(u2).all())}
                if rank == 0 and mode == "bf16":
                    _, _, nprof = timed_loop(step_ncsn, 1, 0, profile="hbm", local=True)
                    hbm_entry("ncsn_prep", f"k_prep (NCSN {ver}: normalise + ELU + bf16 cast of a convolution input)", nprof["ncsn_prep"],
                              f"{nseg} segments: 4 B read + 2 B written per element")
                    hbm_entry("ncsn_pool_resize", f"k_pool5_1d / k_avgpool2 / k_resize2x_add (NCSN {ver})", nprof["ncsn_pool_resize"],
                              f"{nseg} segments: one read + one write of the tensor per pooling / resize")
                ncsn.setdefault(ver, {})[mode] = leg
                del s1, s2

    # ---- 5. Glow training step (config 2): tcgen05 path, per-GPU batch (weak) and the reference's GLOBAL batch 32 (strong)
    train = None
    if args.train_batch > 0:
        from audiosourcesep_b200 import train_glow as tg
        tcfg = GlowConfig(K=args.K)
        tprec = _lib.PREC_FP32 if args.train_fp32 else _lib.PREC_BF16
        tm = Glow(tcfg, init_glow_params(tcfg, seed=2, mode="faithful"), precision=tprec, device=local_rank)
        # the reference's own initialisation: QR/LU 1x1, Glorot conv1/conv2, zero conv3, data-dependent ActNorm
        # (flow_builder.py:96-100); identical on every rank (same seed, rank-0-shaped minibatch)
        tm.init_actnorm(torch.as_tensor(synthetic.mel_patches_db(args.train_batch, seed=300)).to(dev))
        tm.enable_training()
        opt = dict(kind="adamax", lr=1e-3, beta1=0.9, beta2=0.999, eps=1e-7)
        train = {}
        cases = [("weak", args.train_batch, args.train_batch * world)]
        if world > 1 and args.train_batch % world == 0:
            cases.append(("strong", args.train_batch // world, args.train_batch))
        for name, local, glob in cases:
            xt = torch.as_tensor(synthetic.mel_patches_db(glob, seed=300)[rank * local:(rank + 1) * local]).to(dev)
            hist = []

            def step_train():
                hist.append(tg.distributed_train_step(tm, opt, xt, glob))

            nst = max(2, args.steps // 3)
            t_ms, t_launches, _ = timed_loop(step_train, nst, 3)     # eager (sizes the scratch), graph capture, first replay
            losses = [float(v.item()) for v in hist]
            train[name] = {"metric": "glow_train_samples_per_s", "value": glob * nst / (t_ms * 1e-3), "unit": "samples/s",
                           "steps_per_s": nst / (t_ms * 1e-3), "per_gpu_batch": local, "global_batch": glob,
                           "dtype": "f32" if args.train_fp32 else "bf16", "ms_per_step": t_ms / nst, "gpu_launches_per_step": t_launches // nst,
                           "allreduce_bytes_per_step": int(tm.num_trainable * 4) if world > 1 else 0,
                           "alg_tflops": glob * nst * 3 * F_GLOW * (args.K / 40.0) / (t_ms * 1e-3) / 1e12,
                           "step_roofline_frac": glob * nst * 3 * F_GLOW * (args.K / 40.0) / (t_ms * 1e-3) / 1e12 / world / peaks["bf16_sustained"],
                           "loss_first": losses[0], "loss_last": losses[-1], "loss_finite": bool(np.all(np.isfinite(losses))),
                           "loss_decreased": bool(losses[-1] < losses[0])}
        # the same step at a batch that fills the 148 SMs (the reference's batch 32 leaves blocks 2 / 3 of the flow at 96 / 24
        # tiles per launch): how far the kernel path itself goes when it is not tile-starved
        if world == 1 and args.train_big_batch > args.train_batch:
            try:
                nb = args.train_big_batch
                xb_ = torch.as_tensor(synthetic.mel_patches_db(nb, seed=301)).to(dev)
                timed_loop(lambda: tg.distributed_train_step(tm, opt, xb_, nb), 1, 3)
                tb_ms, tb_launches, _ = timed_loop(lambda: tg.distributed_train_step(tm, opt, xb_, nb), 3, 0)
                tfb = nb * 3 * 3 * F_GLOW * (args.K / 40.0) / (tb_ms * 1e-3) / 1e12
                train["big_batch"] = {"metric": "glow_train_samples_per_s", "value": nb * 3 / (tb_ms * 1e-3), "unit": "samples/s",
                                      "per_gpu_batch": nb, "ms_per_step": tb_ms / 3, "alg_tflops": tfb,
                                      "step_roofline_frac": tfb / peaks["bf16_sustained"],
                                      "note": "not the reference's configuration (batch 32): shows the tile-occupancy limit of the small batch"}
                del xb_
            except Exception as ex:          # (never lets an auxiliary leg take the line down)
                train["big_batch"] = {"error": str(ex)[:200]}
        train["note"] = ("tcgen05 forward / data-gradient / weight-gradient GEMMs (bf16 operands, fp32 accumulate), fp32 master weights + "
                         "Adamax, tile images rebuilt on the device every step, gradient pass replayed as a CUDA graph; NCCL all-reduce of "
                         "the flat gradient vector; the loss is that of the reference's own (quirk Q1/Q7) initialisation on synthetic patches")
        del tm

    # ---- 5b. NCSN denoising-score-matching train step (SURVEY 8(f)2; train_ncsn.py:26-57): v1 at the reference's batch 32
    ncsn_train = None
    if args.ncsn_train_batch > 0:
        from audiosourcesep_b200 import NCSNConfig
        from audiosourcesep_b200 import train_ncsn as tn
        from audiosourcesep_b200.ncsn.score_model import ScoreModel
        from audiosourcesep_b200.weights import init_ncsn_params
        ncsn_train = {}
        for ver, ncfg, gflop in (("v1", NCSNConfig(version="v1", ngf=192, num_classes=10, sigma1=1.0), 266.96),
                                 ("v2", NCSNConfig(version="v2", ngf=128, num_classes=200, sigma1=30.0), 118.66)):
            sig_n = bo.get_sigmas(ncfg.sigma1, ncfg.sigmaL, ncfg.num_classes, "logarithmic")
            sm = ScoreModel(ncfg, init_ncsn_params(ncfg, seed=11, mode="faithful"), sigmas=sig_n, device=local_rank, precision=_lib.PREC_BF16)
            sm.enable_training()
            nopt = dict(kind="adam", lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-7)
            cases = [("weak", args.ncsn_train_batch, args.ncsn_train_batch * world)]
            if world > 1 and args.ncsn_train_batch % world == 0:
                cases.append(("strong", args.ncsn_train_batch // world, args.ncsn_train_batch))
            legs = {}
            for name, local, glob in cases:
                xs = torch.as_tensor(synthetic.normalise(synthetic.mel_patches_db(glob, seed=400))[rank * local:(rank + 1) * local]).to(dev)
                gen = torch.Generator(device=dev)
                gen.manual_seed(5)                       # same noise level on every rank and step size class: comparable losses
                hist = []

                def step_nt():
                    idx, z = tn.get_noise_conditionned_data(xs, ncfg.num_classes, gen)
                    hist.append(tn.distributed_train_step(sm, nopt, xs, glob, idx, z))

                nst = max(2, args.steps // 3)
                t_ms, t_launches, _ = timed_loop(step_nt, nst, 2)
                losses = [float(v.item()) for v in hist]
                tf = glob * nst * 3 * gflop / (t_ms * 1e-3) / 1e3
                legs[name] = {"metric": f"ncsn_{ver}_train_samples_per_s", "value": glob * nst / (t_ms * 1e-3), "unit": "samples/s",
                              "steps_per_s": nst / (t_ms * 1e-3), "per_gpu_batch": local, "global_batch": glob, "dtype": "bf16",
                              "ms_per_step": t_ms / nst, "gpu_launches_per_step": t_launches // nst,
                              "allreduce_bytes_per_step": int(sm.num_trainable * 4) if world > 1 else 0,
                              "alg_tflops": tf, "step_roofline_frac": tf / world / peaks["bf16_sustained"],
                              "loss_finite": bool(np.all(np.isfinite(losses)))}
            ncsn_train[ver] = legs
            del sm
        ncsn_train["note"] = ("denoising score matching: forward, data-gradient (k_conv_tc on transposed images) and weight-gradient "
                              "(k_conv_wgrad_tc) convolutions on tcgen05 with bf16 operands, fp32 master weights + Adam, tile images "
                              "rebuilt on the device every step; 3 x score-network FLOPs per sample; one noise level per replica "
                              "batch (train_ncsn.py:34 quirk); parity of the gradients vs float64 autograd: tests/test_gpu_ncsn_train.py")

    # ---- 6. strong scaling of the BASIS configs: the reference's n_mixed = 30 segments SHARDED over the ranks (configs 3-5)
    strong = None
    if world > 1 and args.strong:
        strong = {}
        n_mixed = 30
        lo, hi = (rank * n_mixed) // world, ((rank + 1) * n_mixed) // world
        nloc = hi - lo
        mixed, _, _ = synthetic.basis_problem(n_mixed)
        x1, x2 = synthetic.langevin_init(n_mixed, seed=4)
        bcfg = GlowConfig(K=args.K, minval=0.0, maxval=1.0)
        sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
        eta, lam, ns = bo.langevin_step_constants(sig, 9)
        for mode in [m for m in args.basis_modes.split(",") if m]:
            m1 = Glow(bcfg, init_glow_params(bcfg, seed=2), precision=_prec(_lib, mode), device=local_rank)
            m2 = Glow(bcfg, init_glow_params(bcfg, seed=3), precision=_prec(_lib, mode), device=local_rank)
            md = torch.as_tensor(mixed[lo:hi]).to(dev)
            t1, t2 = torch.as_tensor(x1[lo:hi]).to(dev), torch.as_tensor(x2[lo:hi]).to(dev)
            cnt = [0]

            def step_sb():
                if nloc > 0:
                    ops.basis_glow_inner(m1, m2, md, t1, t2, args.basis_T, float(eta), float(lam), float(ns), seed=1, step0=cnt[0],
                                         elem_offset=lo * D_PATCH)
                cnt[0] += args.basis_T

            nsteps = max(2, args.steps // 2)
            b_ms, _, _ = timed_loop(step_sb, nsteps, 3)
            strong[f"basis_glow_{mode}"] = {"value": n_mixed * args.basis_T * nsteps / (b_ms * 1e-3), "unit": "segment-steps/s",
                                            "n_mixed_total": n_mixed, "segments_this_rank": nloc, "ms_per_langevin_step": b_ms / (nsteps * args.basis_T)}
            del m1, m2
        strong["note"] = ("the reference's n_mixed = 30 segments sharded over the ranks (strong scaling: the N = 1 line's `basis.<mode>.segments.30` "
                          "is the single-GPU figure of the same workload); `train.strong` is the reference's global batch 32 split over the ranks")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # DRAM traffic of the dominant kernel: measured once under `ncu --set full` (profiles/, a committed capture), scaled
    # to this run's launch size -- a constant from a file, labelled as such
    prof_path = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(prof_path):
        try:
            with open(prof_path) as f:
                prof_js = json.load(f)
            per_row = prof_js.get("dram_bytes_per_pixel_row")
            rows_per_launch = B * (48 * 32 + 24 * 16 + 12 * 8) / 3.0
            roofline["traffic"] = None if per_row is None else per_row * rows_per_launch
            roofline["traffic_source"] = ("profiles constant: ncu dram__bytes_read+write per pixel row of a captured block-1 launch "
                                          "(profiles/ncu_summary.json) x mean rows per launch of this run; not measured in this run")
        except Exception:
            pass
    hbm_path = os.path.join(ROOT, "profiles", "r02_hbm_kernels.json")
    if os.path.exists(hbm_path):
        try:
            with open(hbm_path) as f:
                hj = json.load(f)
            for e in roofline_hbm:
                rec = hj.get(e["category"])
                if rec:
                    e["traffic"] = rec["traffic_over_algorithmic"] * e["algorithmic_bytes_per_launch"]
                    e["traffic_source"] = ("profiles constant: dram__bytes_read+write / algorithmic bytes of one `ncu --set full` capture "
                                           f"({rec['capture']}; profiles/r02_hbm_kernels.json) x the algorithmic bytes per launch of this run; "
                                           "not measured in this run")
        except Exception:
            pass

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and args.cpu_sample > 0:
        import torch as _t
        _, probe = cpu_log_prob_rate(2, args.K)                      # size the sample for ~15 s of CPU work
        args.cpu_sample = int(min(64, max(args.cpu_sample, round(15.0 / (probe / 2.0)))))
        rate, secs = cpu_log_prob_rate(args.cpu_sample, args.K)
        cpu = {"value": rate, "unit": "samples/s", "cores": _t.get_num_threads(), "kind": "port",
               "sample": f"{args.cpu_sample} patches, one pass of the reference-faithful graph (coupling network evaluated "
                         f"twice as in the TFP graph), torch-CPU fp32, {secs:.1f} s on {_t.get_num_threads()} threads "
                         f"({os.cpu_count()} logical cores)"}

    line = {
        "metric": "glow_log_prob_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": _config(args, per_gpu_batch=B),
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(x_host.numel() * 4),
                "d2h_bytes_per_step": int(B * 4), "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "roofline_hbm": roofline_hbm,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "alg_tflops": value * F_GLOW * (args.K / 40.0) / 1e12,
        "gate": {"log_prob_nats_per_dim": 1e-3, "measured": None if parity is None or "bf16" not in parity else parity["bf16"]["log_prob_err_nats_per_dim"]},
        "sweep": sweep,
        "directions": directions,
        "basis": basis,
        "basis_ncsn": ncsn or None,
        "train": train,
        "ncsn_train": ncsn_train,
        "strong": strong,
        "parity": parity,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--batch", type=int, default=2048, help="patches per GPU per step")
    ap.add_argument("--K", type=int, default=40, help="flow steps per block (40 = configs/melspec_glow.yml)")
    ap.add_argument("--sweep", type=str, default="30,32,256,4096", help="extra log_prob batch sizes (the headline batch is --batch)")
    ap.add_argument("--modes", type=str, default="bf16,bf16x2,fp16x3", help="Glow precision modes of the inverse / grad_log_prob legs")
    ap.add_argument("--basis-segments", type=str, default="30,256", help="segments per GPU of the Glow-BASIS legs ('' = skip)")
    ap.add_argument("--basis-modes", type=str, default="bf16,fp16x3", help="Glow precision modes of the BASIS legs")
    ap.add_argument("--basis-T", type=int, default=8, help="Langevin steps per library call (steps 2..T replay one CUDA graph)")
    ap.add_argument("--no-parity", dest="parity", action="store_false", help="skip the in-run gate measurements")
    ap.add_argument("--no-strong", dest="strong", action="store_false", help="skip the strong-scaling legs (N > 1)")
    ap.add_argument("--ncsn-modes", type=str, default="bf16,bf16x3")
    ap.add_argument("--ncsn-segments", type=int, default=30, help="segments per GPU of the NCSN-BASIS legs (0 = skip)")
    ap.add_argument("--ncsn-T", type=int, default=8)
    ap.add_argument("--train-batch", type=int, default=32, help="per-GPU batch of the Glow train-step leg (0 = skip)")
    ap.add_argument("--train-big-batch", type=int, default=128, help="auxiliary Glow train leg at a GPU-filling batch (N = 1 only; 0 = skip)")
    ap.add_argument("--ncsn-train-batch", type=int, default=32, help="per-GPU batch of the NCSN train-step legs (0 = skip)")
    ap.add_argument("--train-fp32", action="store_true", help="train leg in the CUDA-core fp32 exact mode")
    ap.add_argument("--cpu-sample", type=int, default=4, help="patches of the CPU baseline sample (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the log-probabilities of the last timed step to DIR/log_prob.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
