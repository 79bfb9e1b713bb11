"""NCSN training -- host-side mirror of the reference's ``train_ncsn.py``.

Same step structure (reference: train_ncsn.py:26-57): ``get_noise_conditionned_data`` draws the noise level and the
perturbation, ``compute_train_loss`` = 1/2 ||scores - target||^2 * sigma^2 averaged over the GLOBAL batch, gradients of
every trainable variable, Adam (train_utils.py:27-28), data-parallel replicas whose gradients are summed.  Here a
replica is one process per GPU (``torchrun``); ``train_grads`` and ``adam_step`` run in libasep.so (forward, data-gradient
and weight-gradient convolutions on tcgen05), the SUM over replicas is one NCCL all-reduce of the flat gradient vector.

Quirk kept (train_ncsn.py:34): ``local_batch_size = X.shape[-1]`` is the CHANNEL count of the NHWC batch, so with the
1-channel mel patches of the configs one noise level (and one Embedding row) is drawn per replica batch and broadcast
over it.  ``--per_sample_sigma`` draws one level per sample instead (the upstream NCSN behaviour).
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
from .config import NCSNConfig, get_config
from .ncsn.utils import get_sigmas


def setUp_optimizer(mirrored_strategy, args):
    """reference: train_utils.py:23-41 (Keras defaults beta1 0.9, beta2 0.999, epsilon 1e-7)."""
    kind = getattr(args, "optimizer", "adam")
    if kind not in ("adam", "adamax"):
        raise ValueError("optimizer argument should be adam or adamax")            # train_utils.py:31-32
    if kind != "adam":
        raise NotImplementedError("the score-network train step implements Adam (the reference's default, train_ncsn.py:405)")
    return dict(kind=kind, lr=float(args.learning_rate), beta1=0.9, beta2=0.999, eps=1e-7)


def get_noise_conditionned_data(X: torch.Tensor, num_classes: int, generator: torch.Generator, per_sample: bool = False):
    """reference: train_ncsn.py:33-44.  Returns (sigma_idx [local batch] int32, z standard normal like X); the
    perturbation ``X + sigmas[idx] * z``, the target ``-z / sigma`` and the weight ``sigma^2`` are applied inside the
    library.  ``local_batch_size = X.shape[-1]`` (:34) is reproduced unless ``per_sample``."""
    n_levels = X.shape[0] if per_sample else X.shape[-1]
    idx = torch.randint(0, int(num_classes), (n_levels,), generator=generator, device=generator.device, dtype=torch.int64)
    if n_levels != X.shape[0]:
        if n_levels != 1:
            raise ValueError("sigma_idx of shape [C] only broadcasts over the batch when C == 1 (train_ncsn.py:34-37)")
        idx = idx.repeat(X.shape[0])
    z = torch.randn(X.shape, generator=generator, device=generator.device, dtype=torch.float32)
    return idx.to(torch.int32), z


def distributed_train_step(model, optimizer: dict, batch: torch.Tensor, global_batch: int, sigma_idx: torch.Tensor,
                           z: torch.Tensor) -> torch.Tensor:
    """One synchronous data-parallel step (reference: train_ncsn.py:46-62); returns the global loss
    (strategy.reduce(SUM) of the per-replica losses)."""
    grads, loss = model.train_grads(batch, z, sigma_idx, global_batch)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(grads, op=dist.ReduceOp.SUM)        # the implicit all-reduce of optimizer.apply_gradients
        dist.all_reduce(loss, op=dist.ReduceOp.SUM)
    model.apply_gradients(grads, optimizer)
    return loss


def shard(perm: np.ndarray, it: int, global_batch: int, rank: int, world: int) -> np.ndarray:
    """Indices of this rank's slice of global batch ``it`` (contiguous blocks, like the Glow trainer)."""
    local = global_batch // world
    return perm[it * global_batch + rank * local: it * global_batch + (rank + 1) * local]


def held_out_dsm(model, sigmas, test: np.ndarray, batch: int, seed: int = 0) -> float:
    """The denoising-score-matching loss of the (normalised) test patches in the units of the train loss, from forward
    score evaluations only: one noise level per patch and z ~ N(0, 1), both drawn from fixed keys (seed, global sample
    index), so every epoch is evaluated on the same perturbations.  Per patch 1/2 sum (score - target)^2 sigma^2 =
    1/2 sum (score sigma + z)^2 (train_ncsn.py:26-44)."""
    from . import ops
    from .train_glow import held_out_mean
    idx_all = np.random.default_rng(seed).integers(0, len(sigmas), test.shape[0]).astype(np.int32)
    sig = torch.as_tensor(np.asarray(sigmas, dtype=np.float32), device=model.device)

    def dsm(x, first):
        idx = torch.as_tensor(idx_all[first: first + x.shape[0]], device=model.device)
        per = int(np.prod(x.shape[1:]))
        z = ops.philox_normal(tuple(x.shape), seed=seed, step=0, stream_id=5, elem_offset=first * per)
        s = sig[idx.long()].reshape(-1, *([1] * (x.ndim - 1)))
        score = model.score(x + s * z, idx)
        return 0.5 * ((score * s + z) ** 2).sum(dim=tuple(range(1, x.ndim)))
    return held_out_mean(test, batch, dsm)


def train(model, optimizer, data: np.ndarray, args, log=print, ema_decay: Optional[float] = None,
          test: Optional[np.ndarray] = None, sigmas=None):
    """Epoch loop over a host dataset of NORMALISED patches (reference: train_ncsn.py:95-160 without the TensorBoard /
    sample-grid side outputs); stops on a NaN / Inf loss (:113-117).  ``ema_decay``: tfa MovingAverage(0.999) of the
    flat parameter vector (train_ncsn.py:327-329), returned as the second value.  ``test``: held-out normalised
    patches; when non-empty, ``Epoch NNN: Test Loss: ...`` (:func:`held_out_dsm` at the noise levels ``sigmas``) is logged
    after every epoch."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    gb = int(args.batch_size)
    if gb % world:
        raise ValueError("batch_size must be divisible by the number of replicas")
    steps_per_epoch = data.shape[0] // gb
    if steps_per_epoch == 0:
        raise ValueError(f"the dataset holds {data.shape[0]} patches, fewer than one global batch of {gb}")
    gen = torch.Generator(device=model.device)
    gen.manual_seed(int(getattr(args, "seed", 0)) * 1000 + rank)
    ema = model.get_flat().clone() if ema_decay else None
    t0, history = time.time(), []
    for epoch in range(int(args.n_epochs)):
        perm = np.random.default_rng(1000 + epoch).permutation(data.shape[0])
        for it in range(steps_per_epoch):
            batch = torch.as_tensor(data[shard(perm, it, gb, rank, world)]).to(model.device)
            idx, z = get_noise_conditionned_data(batch, model.cfg.num_classes, gen, bool(getattr(args, "per_sample_sigma", False)))
            loss = float(distributed_train_step(model, optimizer, batch, gb, idx, z).item())
            history.append(loss)
            if ema is not None:
                ema.mul_(ema_decay).add_(model.get_flat(), alpha=1.0 - ema_decay)
            if not np.isfinite(loss):
                log("Nan or Inf Loss: {}".format(loss))
                return history, ema
        log("Epoch {:03d}: Train Loss: {:.3f}  ({:.1f} s)".format(epoch, float(np.mean(history[-steps_per_epoch:])), time.time() - t0))
        if test is not None and test.shape[0] > 0:
            tl = held_out_dsm(model, sigmas, test, gb // world, seed=int(getattr(args, "seed", 0)))
            log("Epoch {:03d}: Test Loss: {:.6f}".format(epoch, tl))
    return history, ema


def build_parser():
    p = argparse.ArgumentParser(description="Train NCSN model (data-parallel, one process per GPU)")
    p.add_argument("--config", type=str, default=None)
    p.add_argument("--output", type=str, default="trained_ncsn")
    p.add_argument("--version", type=str, default="v2")
    p.add_argument("--ema", action="store_true")
    p.add_argument("--n_train", type=int, default=256, help="synthetic training patches (ignored with --dataset)")
    p.add_argument("--dataset", type=str, default=None,
                   help=".npz of dB mel patches written by audiosourcesep_b200.datasets.wav_to_spec: train on 'train' "
                        "(normalised (x + 100) / 120), log the test loss of 'test' after every epoch")
    p.add_argument("--height", type=int, default=96)
    p.add_argument("--width", type=int, default=64)
    p.add_argument("--n_filters", type=int, default=192)
    p.add_argument("--sigma1", type=float, default=55.0)
    p.add_argument("--sigmaL", type=float, default=0.01)
    p.add_argument("--num_classes", type=int, default=325)
    p.add_argument("--progression", type=str, default="geometric")
    p.add_argument("--n_epochs", type=int, default=1)
    p.add_argument("--optimizer", type=str, default="adam")
    p.add_argument("--batch_size", type=int, default=32)
    p.add_argument("--learning_rate", type=float, default=1e-3)
    p.add_argument("--per_sample_sigma", action="store_true")
    p.add_argument("--exact", action="store_true", help="split-bf16 (three tcgen05 products per GEMM) instead of one")
    p.add_argument("--seed", type=int, default=0)
    return p


def main(args):
    from . import synthetic
    from .ncsn.score_model import ScoreModel
    from .weights import init_ncsn_params
    if args.config is not None:
        for k, v in vars(get_config(args.config)).items():
            setattr(args, k, v)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cfg = NCSNConfig(version=args.version, H=int(args.height), W=int(args.width), ngf=int(args.n_filters),
                     num_classes=int(args.num_classes), sigma1=float(args.sigma1), sigmaL=float(args.sigmaL),
                     progression=args.progression)
    sigmas = get_sigmas(cfg.sigma1, cfg.sigmaL, cfg.num_classes, progression=cfg.progression)
    test = None
    if getattr(args, "dataset", None):
        from .datasets.wav_to_spec import load_patches
        train_db, test_db = load_patches(args.dataset, cfg.H, cfg.W)
        data, test = synthetic.normalise(train_db), synthetic.normalise(test_db)
    else:
        data = synthetic.normalise(synthetic.mel_patches_db(int(args.n_train), int(args.seed), cfg.H, cfg.W))
    model = ScoreModel(cfg, init_ncsn_params(cfg, seed=int(args.seed), mode="faithful"), sigmas=sigmas, device=local_rank,
                       precision=_lib.PREC_BF16X3 if args.exact else _lib.PREC_BF16)
    model.enable_training()
    optimizer = setUp_optimizer(None, args)
    log = print if rank == 0 else (lambda *a, **k: None)
    log("Total Trainable Variables: ", model.count_params())
    t0 = time.time()
    hist, ema = train(model, optimizer, data, args, log=log, ema_decay=0.999 if args.ema else None, test=test, sigmas=sigmas)
    log("Training time: ", np.round(time.time() - t0, 2), " seconds")
    if rank == 0:
        if ema is not None:
            model.set_flat(ema)
        model.sync_host()
        os.makedirs(args.output, exist_ok=True)
        np.savez(os.path.join(args.output, "weights.npz"), **model.variables)
    return hist


if __name__ == "__main__":
    main(build_parser().parse_args())
