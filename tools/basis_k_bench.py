"""BASIS with K sources on one GPU: ms per Langevin step and throughput of the K-source step, and the fused K-source update
kernel alone.

    python tools/basis_k_bench.py --out <dir>

1. One Langevin step of K = 2, 3, 4 sources at the reference's n_mixed = 30 segments and T = 8 steps per library call (the
   bench.py defaults; steps 2..T replay one CUDA graph): Glow bf16 and fp16x3 priors of full depth (K_flow = 40), NCSN v1
   and v2 score networks in bf16.  Each row is CUDA events around `calls` calls after 3 warm-up calls.  A segment-step is
   one update of all K sources of one segment; source-steps/s = segment-steps/s x K.  Glow bf16 also runs with ONE handle
   serving every source (its K score evaluations one after another on one branch of the step graph) next to K distinct
   handles (K parallel branches): both rows do the same arithmetic, so their ratio is what the parallel branches buy.
2. The K-source update kernel alone (asep_langevin_step_k) at 4096 segments, K = 2, 3, 4, with in-kernel Philox noise and
   with injected noise: (3K+1) x 4 B / (4K+1) x 4 B of algorithmic traffic per element (every tensor is 100 MB, the working
   set is larger than the 126 MB L2) over event time, and its fraction of the 6551 GB/s copy peak measured for this
   project (DESIGN.md section 3).
The card's name and power limit are recorded beside the numbers.  Writes <out>/basis_k_bench.json.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from audiosourcesep_b200 import GlowConfig, NCSNConfig, _lib, ops, synthetic  # noqa: E402
from audiosourcesep_b200.glow import Glow  # noqa: E402
from audiosourcesep_b200.ncsn.score_model import ScoreModel  # noqa: E402
from audiosourcesep_b200.weights import init_glow_params, init_ncsn_params  # noqa: E402
from oracle import basis_oracle as bo  # noqa: E402

COPY_PEAK_GBS = 6551.0          # DESIGN.md section 3: measured device-to-device copy rate of the B200 this project runs on


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "unavailable"}


def timed(fn, calls, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def step_rows(kind, models, n_mixed, T, calls, Ks, one_handle=False):
    rows = {}
    for K in Ks:
        mixed, _, _ = synthetic.basis_problem(n_mixed)
        rng = np.random.default_rng(K)
        x = torch.as_tensor(rng.uniform(0, 1, (K, n_mixed, 96, 64, 1)).astype(np.float32)).cuda()
        mixed_d = torch.as_tensor(mixed).cuda()
        ms = [models[0]] * K if one_handle else models[:K]
        step = [0]
        if kind == "glow":
            sig = bo.get_sigmas(1.0, 0.01, 10, "logarithmic")
            eta, lam, ns = bo.step_constants(sig, 9)

            def call():
                ops.basis_glow_inner_k(ms, mixed_d, x, T, float(eta), float(lam), float(ns), seed=1, step0=step[0])
                step[0] += T
        else:
            idx = 3                                           # kind = (name, sigma1, num_classes)
            sig = bo.get_sigmas(kind[1], 0.01, kind[2], "logarithmic")
            eta, lam, ns = bo.step_constants(sig, idx)

            def call():
                ops.basis_ncsn_inner_k(ms, mixed_d, x, idx, T, float(eta), float(lam), float(ns), seed=1, step0=step[0])
                step[0] += T
        ms_total = timed(call, calls)
        ms_step = ms_total / (calls * T)
        rows[str(K)] = {"ms_per_langevin_step": ms_step, "segment_steps_per_s": n_mixed / (ms_step * 1e-3),
                        "source_steps_per_s": K * n_mixed / (ms_step * 1e-3), "timed_steps": calls * T,
                        "finite": bool(torch.isfinite(x).all())}
        print(kind if isinstance(kind, str) else kind[0], "one-handle" if one_handle else "distinct", K, f"{ms_step:.3f} ms/step",
              flush=True)
        del x
    return rows


def kernel_rows(Ks, nseg, reps):
    shp = (nseg, 96, 64, 1)
    n = int(np.prod(shp))
    g = torch.Generator(device="cuda").manual_seed(0)
    mixed = torch.rand(shp, device="cuda", generator=g)
    rows = {}
    for K in Ks:
        x = torch.rand((K,) + shp, device="cuda", generator=g)
        s = torch.randn((K,) + shp, device="cuda", generator=g) * 1e-3
        z = torch.randn((K,) + shp, device="cuda", generator=g)
        for name, noise, per_elem in (("philox", None, (3 * K + 1) * 4), ("injected", z, (4 * K + 1) * 4)):
            ms = timed(lambda: ops.langevin_step_k(x, s, mixed, 2e-5, 1e4, 6.3e-3, noise=noise, seed=1, step=0), reps, 2) / reps
            gbs = per_elem * n / (ms * 1e-3) / 1e9
            rows[f"{K}_{name}"] = {"K": K, "noise": name, "ms_per_launch": ms, "algorithmic_bytes_per_element": per_elem,
                                   "algorithmic_GBps": gbs, "fraction_of_copy_peak": gbs / COPY_PEAK_GBS}
            print("kernel", K, name, f"{ms:.3f} ms {gbs:.0f} GB/s", flush=True)
        del x, s, z
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n_mixed", type=int, default=30)
    ap.add_argument("--T", type=int, default=8)
    ap.add_argument("--calls", type=int, default=4)
    ap.add_argument("--sources", type=str, default="2,3,4")
    ap.add_argument("--kernel_segments", type=int, default=4096)
    args = ap.parse_args()
    _lib.init()
    Ks = [int(v) for v in args.sources.split(",")]
    out = {"card": card(), "n_mixed": args.n_mixed, "T_per_call": args.T, "timed_calls": args.calls,
           "steps": {}, "kernel": None}
    cfg = GlowConfig(K=40, minval=0.0, maxval=1.0)
    for mode, prec in (("bf16", _lib.PREC_BF16), ("fp16x3", _lib.PREC_FP16X3)):
        models = [Glow(cfg, init_glow_params(cfg, seed=2 + k), precision=prec) for k in range(max(Ks))]
        out["steps"][f"glow_{mode}"] = step_rows("glow", models, args.n_mixed, args.T, args.calls, Ks)
        if mode == "bf16":
            out["steps"]["glow_bf16_one_handle"] = step_rows("glow", models, args.n_mixed, args.T, args.calls, Ks, one_handle=True)
        del models
        torch.cuda.empty_cache()
    for ver, ncfg in (("v1", NCSNConfig(version="v1", ngf=192, num_classes=10, sigma1=1.0)),
                      ("v2", NCSNConfig(version="v2", ngf=128, num_classes=200, sigma1=30.0))):
        sig = bo.get_sigmas(ncfg.sigma1, ncfg.sigmaL, ncfg.num_classes, "logarithmic")
        models = [ScoreModel(ncfg, init_ncsn_params(ncfg, seed=11 + k), sigmas=sig, precision=_lib.PREC_BF16)
                  for k in range(max(Ks))]
        out["steps"][f"ncsn_{ver}_bf16"] = step_rows((f"ncsn_{ver}", ncfg.sigma1, ncfg.num_classes), models, args.n_mixed,
                                                     args.T, args.calls, Ks)
        del models
        torch.cuda.empty_cache()
    out["kernel"] = kernel_rows(Ks, args.kernel_segments, 20)
    out["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "basis_k_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
