"""Glow / noisy-Glow training -- host-side mirror of the reference's ``train_glow.py`` and ``train_noisy_glow.py``.

Same step structure (reference: train_glow.py:29-54): ``compute_train_loss`` = sum_i -log_prob(x_i) / global batch,
gradients of every trainable variable, Adamax (train_utils.py:29-30), data-parallel replicas whose gradients are
summed.  Here a replica is one process per GPU (``torchrun``); ``train_grads`` runs in libasep.so, the SUM over
replicas is one NCCL all-reduce of the flat gradient vector over NVLink, ``adamax_step`` runs in libasep.so.
``train_noisy_glow`` adds ``sigma * N(0,1)`` in raw data units before ``log_prob`` (reference:
train_noisy_glow.py:30-33) and walks the noise levels serially, each level warm-started from the previous one and
written to ``<output>/sigma_<round(sigma,2)>/weights.npz`` -- the layout run_basis_sep reads (reference:
train_noisy_glow.py:309-358, run_basis_sep.py:284-285).
"""
from __future__ import annotations

import argparse
import os
import time
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .config import get_config
from .ncsn.utils import get_sigmas


def setUp_optimizer(mirrored_strategy, args):
    """reference: train_utils.py:23-41 -- the Keras Adam / Adamax hyper-parameters (defaults beta1 0.9, beta2 0.999,
    epsilon 1e-7) as the dictionary ``Glow.apply_gradients`` takes; the update itself runs in libasep.so."""
    kind = getattr(args, "optimizer", "adamax")
    if kind not in ("adam", "adamax"):
        raise ValueError("optimizer argument should be adam or adamax")            # train_utils.py:31-32
    return dict(kind=kind, lr=float(args.learning_rate), beta1=0.9, beta2=0.999, eps=1e-7)


def distributed_train_step(flow, optimizer: dict, batch: torch.Tensor, global_batch: int,
                           noise: Optional[torch.Tensor] = None, sigma: float = 0.0) -> torch.Tensor:
    """One synchronous data-parallel step (reference: train_glow.py:37-54).  ``batch`` is this rank's shard; returns
    the global loss (sum of the per-replica losses, strategy.reduce(SUM))."""
    grads, loss = flow.train_grads(batch, global_batch, noise=noise, sigma=sigma)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(grads, op=dist.ReduceOp.SUM)        # NCCL over NVLink: the implicit all-reduce of apply_gradients
        dist.all_reduce(loss, op=dist.ReduceOp.SUM)         # strategy.reduce(SUM, per_replica_losses)
    if hasattr(flow, "apply_gradients"):
        flow.apply_gradients(grads, optimizer)
    else:                                                    # duck-typed handles (tests) with the Adamax-only surface
        flow.adamax_step(grads, **{k: v for k, v in optimizer.items() if k != "kind"})
    return loss


def noise_for(batch_shape, seed: int, step: int, rank_offset: int, device) -> torch.Tensor:
    """Standard normals keyed by (seed, step, global sample index) so that any number of replicas draws the same
    noise for the same global batch."""
    from . import ops
    n = int(np.prod(batch_shape))
    return ops.philox_normal(tuple(batch_shape), seed=seed, step=step, stream_id=3, elem_offset=rank_offset * (n // batch_shape[0]))


def synthetic_dataset(n: int, seed: int, H: int, W: int) -> np.ndarray:
    from . import synthetic
    return synthetic.mel_patches_db(n, seed, H, W)


def held_out_mean(test: np.ndarray, batch: int, per_sample_loss) -> float:
    """Mean of ``per_sample_loss(x, first)`` (a device vector of losses of the test patches ``x`` whose first global
    index is ``first``) over every test patch.  Each rank evaluates one contiguous shard in chunks of ``batch``; the
    float64 sums are all-reduced, so every rank returns the same value."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    n = test.shape[0]
    lo, hi = rank * n // world, (rank + 1) * n // world
    total = torch.zeros((1,), dtype=torch.float64, device=torch.device("cuda", torch.cuda.current_device()))
    for c0 in range(lo, hi, max(1, int(batch))):
        x = torch.as_tensor(test[c0: min(c0 + int(batch), hi)]).to(total.device)
        total += per_sample_loss(x, c0).double().sum()
    if world > 1:
        dist.all_reduce(total, op=dist.ReduceOp.SUM)
    return float(total.item()) / n


def held_out_nll(flow, test: np.ndarray, batch: int, sigma: float = 0.0, seed: int = 0) -> float:
    """Mean -log_prob over the test patches, the units of the train loss; at a noise level ``sigma`` the patches are
    perturbed by sigma * N(0, 1) in raw data units, drawn from a fixed Philox key (seed, global sample index), so the
    test loss of successive epochs is evaluated on the same perturbation."""
    from . import ops

    def nll(x, first):
        if sigma > 0.0:
            per = int(np.prod(x.shape[1:]))
            x = x + float(sigma) * ops.philox_normal(tuple(x.shape), seed=seed, step=0, stream_id=4, elem_offset=first * per)
        return -flow.log_prob(x)
    return held_out_mean(test, batch, nll)


def train(flow, optimizer, data: np.ndarray, args, sigma: float = 0.0, log=print, step_offset: int = 0,
          test: Optional[np.ndarray] = None):
    """Epoch loop over a host dataset (reference: train_glow.py:88-181 without the TensorBoard / sample-grid side
    outputs); stops on a NaN / Inf loss like train_glow.py:115-118.  ``step_offset``: global step of the first
    iteration -- the noise of train_noisy_glow is keyed by (seed, global step, global sample), so successive calls
    (one per noise level) must continue the count instead of redrawing the same sequence.  ``test``: held-out patches;
    when non-empty, ``Epoch NNN: Test Loss: ...`` (:func:`held_out_nll`) is logged after every epoch."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    gb = int(args.batch_size)
    if gb % world:
        raise ValueError("batch_size must be divisible by the number of replicas")
    local = gb // world
    steps_per_epoch = data.shape[0] // gb
    if steps_per_epoch == 0:
        raise ValueError(f"the dataset holds {data.shape[0]} patches, fewer than one global batch of {gb}")
    step, t0, history = int(step_offset), time.time(), []
    for epoch in range(int(args.n_epochs)):
        perm = np.random.default_rng(1000 + epoch).permutation(data.shape[0])
        for it in range(steps_per_epoch):
            idx = perm[it * gb + rank * local: it * gb + (rank + 1) * local]
            batch = torch.as_tensor(data[idx]).to(flow.device)
            noise = None
            if sigma > 0.0:
                noise = noise_for(batch.shape, seed=int(getattr(args, "seed", 0)), step=step, rank_offset=rank * local,
                                  device=flow.device)
            loss = float(distributed_train_step(flow, optimizer, batch, gb, noise=noise, sigma=sigma).item())
            history.append(loss)
            if not np.isfinite(loss):
                log("NaN / Inf loss at step {}: stopping".format(step))
                return history
            step += 1
        log("Epoch {:03d}: loss = {:.4f}  ({:.1f} s)".format(epoch, history[-1], time.time() - t0))
        if test is not None and test.shape[0] > 0:
            tl = held_out_nll(flow, test, local, sigma=sigma, seed=int(getattr(args, "seed", 0)))
            log("Epoch {:03d}: Test Loss: {:.6f}".format(epoch, tl))
    return history


def build_parser():
    p = argparse.ArgumentParser(description="Train Glow (data-parallel, one process per GPU)")
    p.add_argument("--config", type=str, default=None)
    p.add_argument("--output", type=str, default="trained_glow")
    p.add_argument("--n_train", type=int, default=256, help="synthetic training patches (ignored with --dataset)")
    p.add_argument("--dataset", type=str, default=None,
                   help=".npz of dB mel patches written by audiosourcesep_b200.datasets.wav_to_spec: train on 'train', "
                        "log the test loss of 'test' after every epoch")
    p.add_argument("--height", type=int, default=96)
    p.add_argument("--width", type=int, default=64)
    p.add_argument("--L", type=int, default=3)
    p.add_argument("--K", type=int, default=40)
    p.add_argument("--n_filters", type=int, default=512)
    p.add_argument("--learntop", action="store_true", default=True)
    p.add_argument("--n_epochs", type=int, default=1)
    p.add_argument("--batch_size", type=int, default=32)
    p.add_argument("--learning_rate", type=float, default=1e-3)
    p.add_argument("--optimizer", type=str, default="adamax")
    p.add_argument("--noisy", action="store_true", help="train_noisy_glow: fine-tune one model per noise level")
    p.add_argument("--sigma1", type=float, default=1.0)
    p.add_argument("--sigmaL", type=float, default=0.01)
    p.add_argument("--num_classes", type=int, default=10)
    p.add_argument("--progression", type=str, default="logarithmic")
    p.add_argument("--seed", type=int, default=0)
    return p


def main(args):
    from .flow_models.flow_builder import build_glow
    if args.config is not None:
        for k, v in vars(get_config(args.config)).items():
            setattr(args, k, v)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    test = None
    if getattr(args, "dataset", None):
        from .datasets.wav_to_spec import load_patches
        data, test = load_patches(args.dataset, args.height, args.width)
    else:
        data = synthetic_dataset(int(args.n_train), int(args.seed), args.height, args.width)
    minibatch = data[: int(args.batch_size)]                     # data-dependent ActNorm init batch (train_glow.py:300-306)
    flow = build_glow(minibatch, [args.height, args.width, 1], L=args.L, K=args.K, n_filters=args.n_filters,
                      learntop=args.learntop, l2_reg=None, data_type="melspec", minval=-100.0, maxval=20.0,
                      use_logit=False, seed=int(args.seed), precision=_lib.PREC_BF16 if int(args.n_filters) == 512 else None)
    flow.enable_training()
    optimizer = setUp_optimizer(None, args)
    log = print if rank == 0 else (lambda *a, **k: None)
    if not args.noisy:
        hist = train(flow, optimizer, data, args, log=log, test=test)
        if rank == 0:
            flow.sync_host()
            os.makedirs(args.output, exist_ok=True)
            np.savez(os.path.join(args.output, "weights.npz"), **flow.variables)
        return hist
    sigmas = get_sigmas(args.sigma1, args.sigmaL, int(args.num_classes), progression=args.progression)
    hist = []
    for sigma in sigmas:                                         # serial over noise levels, warm start (train_noisy_glow.py:309-358)
        log("Training at noise level sigma = {}".format(sigma))
        # noise is added in RAW data units (dB), train_noisy_glow.py:31-32
        hist += train(flow, optimizer, data, args, sigma=float(sigma), log=log, step_offset=len(hist), test=test)
        if rank == 0:
            flow.sync_host()
            d = os.path.join(args.output, "sigma_" + str(round(float(sigma), 2)))
            os.makedirs(d, exist_ok=True)
            np.savez(os.path.join(d, "weights.npz"), **flow.variables)
    return hist


if __name__ == "__main__":
    main(build_parser().parse_args())
