"""BASIS separation driver -- host-side mirror of the reference's ``run_basis_sep.py``.

Same entry points (``compute_grad_logprob``, ``mixing_process``, ``post_processing_fn``,
``basis_inner_loop``, ``basis_outer_loop``, ``main``), same CLI flags and the same outputs
(``results.npz`` with x1/x2/gt1/gt2/mixed/stft_mixture, ``results_convergence.npz`` with the per-sigma
snapshots, ``out.log`` with the "Sigma = ..." / "Duration: ... seconds" lines that downstream readers
parse; reference: run_basis_sep.py:73-260, :263-450, :453-525).  The arithmetic of the loop -- both
score evaluations, the mixture-consistency gradient, the noise injection and the state update -- runs in
libasep.so; Python only sequences noise levels.

Differences from the shipped script, all forced by its defects (SURVEY.md App. D, D1/D2/D7):
* ``--config`` values are laid over the argparse defaults instead of replacing them, so keys missing from
  the YAML (``T``, ``version``, ``l2_reg``) keep their defaults;
* the Glow branch builds its priors from ``data_shape`` with ``SpecPreprocessing(minval=0, maxval=1)``
  because BASIS states live in normalised [0, 1] units (SURVEY.md App. B);
* weights come from ``.npz`` containers (``<RESTORE>/sigma_<round(sigma,2)>/weights.npz`` for Glow,
  ``<RESTORE>/weights.npz`` for NCSN) or, with ``--random_init SEED``, from the seeded generators -- the
  reference ships no checkpoint and TensorFlow bundles cannot be read here;
* mel patches come from ``<song_dir>/{mix,piano,violin}.wav`` through the GPU front end (datasets/data_loader.py:
  get_song_extract, as in the reference), from ``<song_dir>/{mix,piano,violin}.npy`` (dB, ``[n,96,64]``), or are generated
  with ``--synthetic``.

Beyond the reference, K = 2..8 sources are separated: one prior per restore directory (``RESTORE1 RESTORE2 [RESTORE ...]``,
all of one ``model_type``), the stems named by ``--sources`` (``piano,violin`` by default, for K = 2), and
``results.npz`` / ``results_convergence.npz`` holding ``x1..xK`` (and ``gt1..gtK``).  The loop works on one stacked state
``[K, n, H, W, 1]`` (basis_inner_loop_k / basis_outer_loop_k); the two-source functions are its K = 2 case.

``--mix PATH`` separates a whole recording from its mixture alone (track.py): the wav file is cut into overlapping 2.04 s
segments (``--overlap_frames``, default 8), nothing skipped or dropped; ``results.npz`` then holds x1..xK / mixed /
stft_mixture over all segments plus ``segment_start``, ``track_length``, ``orig_sr``, ``orig_length`` and
``overlap_frames`` (no gt keys), and rank 0 writes ``<output>/<source name>.wav`` at the input's rate and length and
``separated.npz`` with the float32 tracks.  ``--render mask [--mwf_iterations N]`` makes those stems as multichannel Wiener
masks on the recording itself instead (track.render_track): they keep its channels and full band and sum to it.

Segments are independent (SURVEY.md 8(e)): under ``torchrun`` every rank separates a contiguous block of
segments with noise keyed by the GLOBAL element index, and rank 0 gathers the blocks at the end -- the
only cross-GPU traffic.
"""
from __future__ import annotations

import argparse
import os
import sys
import time
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np

from .config import GlowConfig, NCSNConfig, get_config
from .ncsn.utils import get_sigmas, langevin_step_constants

D_MIN, D_MAX = -100.0, 20.0


# --------------------------------------------------------------------------------------- sharding
def shard_range(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous block of ceil(n/world) segments for ``rank`` (SURVEY.md 8(e))."""
    per = (n + world - 1) // world
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def gather_segments(local: np.ndarray, n_total: int, axis: int = 0) -> Optional[np.ndarray]:
    """Gather the per-rank segment blocks on rank 0 (returns None elsewhere).  Uses the default process
    group if one is initialised (NCCL on GPUs, gloo in the CPU tests); a single process returns ``local``."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local
    world, rank = dist.get_world_size(), dist.get_rank()
    parts: List[Optional[np.ndarray]] = [None] * world if rank == 0 else None
    dist.gather_object(local, parts, dst=0)
    if rank != 0:
        return None
    out = np.concatenate([p for p in parts if p is not None and p.shape[axis] > 0], axis=axis)
    assert out.shape[axis] == n_total, (out.shape, n_total)
    return out


# --------------------------------------------------------------------------------------- reference API
def compute_grad_logprob(inputs, model):
    """grad_x log p(x) (reference: run_basis_sep.py:73-79)."""
    return model.grad_log_prob(inputs)


def post_processing_fn(args) -> Callable[[np.ndarray], np.ndarray]:
    """reference: run_basis_sep.py:82-96 (melspec branch)."""
    minval, maxval = float(args.minval), float(args.maxval)
    use_logit, alpha = bool(getattr(args, "use_logit", False)), getattr(args, "alpha", 1e-6) or 0.0

    def post_processing(x):
        x = np.asarray(x, dtype=np.float32)
        if use_logit:
            x = 1.0 / (1.0 + np.exp(-x))
            x = (x - alpha) / (1.0 - 2.0 * alpha)
        x = x * (maxval - minval) + minval
        return np.clip(x, minval, maxval)

    return post_processing


def mixing_process(args):
    """(g, grad_g) on device tensors (reference: run_basis_sep.py:106-149).  Only the dB mel-spectrogram
    mixing of the shipped configs runs as a CUDA kernel; the loop itself uses the fused Langevin kernel."""
    from . import ops
    if getattr(args, "data_type", "melspec") != "melspec" or getattr(args, "scale", "dB") != "dB":
        raise NotImplementedError("only the dB mel-spectrogram mixing of configs/melspec_*.yml is on the hot path")

    def g(x1, x2):
        return ops.mixing_db(x1, x2)[0]

    def grad_g(x1, x2):
        _, w1, w2 = ops.mixing_db(x1, x2)
        return w1, w2

    return g, grad_g


def basis_inner_loop_k(mixed, x, models, sigma_idx, sigmas, g=None, grad_g=None, post_processing=None, model_type="ncsn",
                       delta=2e-5, T=100, debug=True, train_summary_writer=None, step=None, noise=None, seed=0,
                       elem_offset=0, per_step=None, **kwargs):
    """T fused Langevin updates of K sources at noise level ``sigma_idx`` (reference: run_basis_sep.py:152-214).

    ``x`` [K, n, H, W, 1] is a CUDA tensor updated IN PLACE and returned; ``models[k]`` is the prior of source k.
    ``noise`` ([T, K, n, H, W, 1] standard normals) injects the draws for parity runs; otherwise Philox noise keyed by
    (seed, global step, global element index) is generated inside the kernel, source k on stream k + 1."""
    import torch
    from . import ops
    eta, lam, ns = langevin_step_constants(sigmas, sigma_idx, delta)
    step0 = int(sigma_idx) * int(T)
    nan = torch.zeros(1, dtype=torch.int32, device=x.device) if debug else None
    if model_type == "glow":
        ops.basis_glow_inner_k(models, mixed, x, int(T), float(eta), float(lam), float(ns), noise=noise, seed=seed,
                               step0=step0, elem_offset=elem_offset, per_step=per_step, nan_count=nan)
    elif all(hasattr(m, "handle") for m in models):
        ops.basis_ncsn_inner_k(models, mixed, x, int(sigma_idx), int(T), float(eta), float(lam), float(ns), noise=noise,
                               seed=seed, step0=step0, elem_offset=elem_offset, per_step=per_step, nan_count=nan)
    else:                                                              # any callable score model (plug-in seam)
        n = x.shape[1]
        idx = torch.full((n,), int(sigma_idx), dtype=torch.int32, device=x.device)
        for t in range(int(T)):
            s = torch.stack([m([x[k], idx], training=True) for k, m in enumerate(models)])   # run_basis_sep.py:167-170
            ops.langevin_step_k(x, s, mixed, float(eta), float(lam), float(ns), noise=None if noise is None else noise[t],
                                seed=seed, step=step0 + t, elem_offset=elem_offset, nan_count=nan)
            if per_step is not None:
                per_step[t].copy_(x)
    if debug and int(nan.item()) != 0:                                 # the reference's --debug NaN asserts, :183-191
        raise FloatingPointError(f"NaN in the Langevin state at sigma index {sigma_idx}")
    return x


def basis_inner_loop(mixed, x1, x2, model1, model2, sigma_idx, sigmas, g=None, grad_g=None, post_processing=None,
                     model_type="ncsn", delta=2e-5, T=100, debug=True, train_summary_writer=None, step=None,
                     noise1=None, noise2=None, seed=0, elem_offset=0, per_step=None, **kwargs):
    """T fused Langevin updates at noise level ``sigma_idx`` (reference: run_basis_sep.py:152-214): basis_inner_loop_k
    with K = 2.

    x1 / x2 are CUDA tensors updated IN PLACE and returned.  ``noise1/noise2`` ([T, n, H, W, 1] standard
    normals) inject the draws for parity runs; otherwise Philox noise keyed by (seed, global step, global
    element index) is generated inside the kernel."""
    import torch
    x = torch.stack([x1, x2])
    noise = None if noise1 is None else torch.stack([torch.as_tensor(noise1), torch.as_tensor(noise2)], 1)
    try:
        basis_inner_loop_k(mixed, x, [model1, model2], sigma_idx, sigmas, model_type=model_type, delta=delta, T=T, debug=debug,
                           noise=noise, seed=seed, elem_offset=elem_offset, per_step=per_step)
    finally:
        x1.copy_(x[0])
        x2.copy_(x[1])
    return x1, x2


def basis_outer_loop_k(mixed, x, models, optimizer, sigmas, ckpts, args, train_summary_writer=None):
    """reference: run_basis_sep.py:217-260 for K sources: ``x`` [K, n, H, W, 1] is updated in place.  ``ckpts[k]`` is a
    callable ``sigma -> params dict or None`` that supplies the per-noise-level Glow weights of prior k (the reference
    restores a checkpoint per sigma, :228-234), or None.  Returns (x, x_arr) with x_arr = {"x1": [...], ..., "xK": [...]}."""
    K = len(models)
    x_arr = {f"x{k + 1}": [x[k].detach().cpu().numpy().copy()] for k in range(K)}
    ckpts = list(ckpts) if ckpts is not None else [None] * K
    device_loop = (not getattr(args, "host_loop", False) and all(hasattr(m, "handle") for m in models)
                   and (args.model_type == "ncsn" or all(c is None for c in ckpts)))
    if device_loop:
        # the whole sigma x T loop inside the library (asep_basis_ncsn_run_k / asep_basis_glow_run_k): no host round trip
        # between noise levels, the per-level snapshots are copied on the stream and read once at the end
        import torch
        from . import ops
        L = len(sigmas)
        consts = [langevin_step_constants(sigmas, i, 2e-5) for i in range(L)]
        snaps = torch.empty((L,) + tuple(x.shape), dtype=torch.float32, device=x.device)
        nan = torch.zeros(1, dtype=torch.int32, device=x.device) if args.debug else None
        for sigma_idx, sigma in enumerate(sigmas):
            print("Sigma = {} ({} / {})".format(sigma, sigma_idx + 1, L))
        ops.basis_run_k(models, mixed, x, int(args.T), [c[0] for c in consts], [c[1] for c in consts], [c[2] for c in consts],
                        seed=getattr(args, "seed", 0), elem_offset=getattr(args, "elem_offset", 0), snapshots=snaps,
                        nan_count=nan)
        if args.debug and int(nan.item()) != 0:
            raise FloatingPointError("NaN in the Langevin state")
        host = snaps.cpu().numpy()
        for i in range(L):
            for k in range(K):
                x_arr[f"x{k + 1}"].append(host[i, k].copy())
        print("inner loop done")
        print("_" * 100)
        return x, x_arr
    for sigma_idx, sigma in enumerate(sigmas):
        print("Sigma = {} ({} / {})".format(sigma, sigma_idx + 1, len(sigmas)))
        if args.model_type == "glow":
            for tag, (m, ck) in enumerate(zip(models, ckpts), start=1):
                p = ck(float(sigma)) if ck is not None else None
                if p is not None:
                    m.set_params(p)
                    m.prepare()
                    print("Model {} at noise level {} restored".format(tag, sigma))
        basis_inner_loop_k(mixed, x, models, sigma_idx, sigmas, model_type=args.model_type, delta=2e-5, T=args.T,
                           debug=args.debug, seed=getattr(args, "seed", 0), elem_offset=getattr(args, "elem_offset", 0))
        for k in range(K):
            x_arr[f"x{k + 1}"].append(x[k].detach().cpu().numpy().copy())
        print("inner loop done")
        print("_" * 100)
    return x, x_arr


def basis_outer_loop(mixed, x1, x2, model1, model2, optimizer, sigmas, ckpt1, ckpt2, args, train_summary_writer=None):
    """reference: run_basis_sep.py:217-260: basis_outer_loop_k with K = 2.  ``ckpt1/ckpt2`` are callables
    ``sigma -> params dict or None`` that supply the per-noise-level Glow weights (the reference restores a checkpoint
    per sigma, :228-234)."""
    import torch
    x = torch.stack([x1, x2])
    try:
        x, x_arr = basis_outer_loop_k(mixed, x, [model1, model2], optimizer, sigmas, [ckpt1, ckpt2], args, train_summary_writer)
    finally:
        x1.copy_(x[0])
        x2.copy_(x[1])
    return x1, x2, x_arr


# --------------------------------------------------------------------------------------- data / weights
def load_song_patches(args):
    """(mixed_db, [gt_1_db, ..., gt_K_db], stft_mixture) as float32 [n_mixed, H, W, 1] in dB, one ground truth per source
    (source_names)."""
    from . import synthetic
    n = int(args.n_mixed)
    names = source_names(args)
    if getattr(args, "synthetic", False) or args.song_dir is None:
        if args.song_dir is None and not getattr(args, "synthetic", False):
            raise ValueError("song_dir is None")                       # run_basis_sep.py:300-301
        gts = [synthetic.mel_patches_db(n, k, args.height, args.width) for k in range(len(names))]
        return synthetic.mixture_db(*gts), gts, np.zeros((n, 1025, args.width), np.complex64)
    d = os.path.abspath(args.song_dir)
    if os.path.exists(os.path.join(d, "mix.wav")):                    # the reference's own input (run_basis_sep.py:342-351)
        from .datasets import data_loader
        spec_params = {"length_sec": 2.04, "dbmin": -100, "dbmax": 20, "fmin": 125, "fmax": 7600, "use_dB": True, "n_fft": 2048,
                       "hop_length": 512, "n_mels": 96, "sr": 16000}
        mel_spec, _, stft_mixture = data_loader.get_song_extract_k(os.path.join(d, "mix.wav"),
                                                                   [os.path.join(d, nm + ".wav") for nm in names], 2.04 * n,
                                                                   **spec_params)
        mix, *gts = (m.cpu().numpy() for m in mel_spec)
        if mix.shape[1:] != (args.height, args.width, 1):
            raise ValueError(f"mel patches of shape {mix.shape[1:]}, the model expects {(args.height, args.width, 1)}")
        return mix, gts, stft_mixture
    arrs = []
    for name in ["mix"] + names:
        a = np.load(os.path.join(d, name + ".npy")).astype(np.float32)
        if a.ndim == 3:
            a = a[..., None]
        if a.shape[0] < n or a.shape[1:] != (args.height, args.width, 1):
            raise ValueError(f"{name}.npy: expected at least {n} patches of {args.height}x{args.width}, got {a.shape}")
        arrs.append(a[:n])
    stft_path = os.path.join(d, "stft_mixture.npy")
    stft = np.load(stft_path)[:n] if os.path.exists(stft_path) else np.zeros((n, 1025, args.width), np.complex64)
    return arrs[0], arrs[1:], stft


def load_mix_patches(args):
    """Whole-track front end of ``--mix`` (track.py): (mixed_db float32 [n_seg, H, W, 1], stft_mixture complex64
    [n_seg, 1025, W], segmentation) with segmentation = segment_start, track_length, orig_sr and orig_length."""
    from . import track
    x, rate, length = track.read_track(os.path.abspath(args.mix))
    mel, stft, starts = track.segment_track(x, args.overlap_frames)
    mix = mel.cpu().numpy()
    if mix.shape[1:] != (args.height, args.width, 1):
        raise ValueError(f"mel patches of shape {mix.shape[1:]}, the model expects {(args.height, args.width, 1)}")
    return mix, stft.cpu().numpy(), {"starts": starts, "track_length": int(x.numel()), "orig_sr": rate, "orig_length": length}


def load_weights(directory: str, shapes: Dict[str, tuple]) -> Dict[str, np.ndarray]:
    """Weights of one model: ``<directory>/weights.npz`` (this package's container) or, failing that, the TensorFlow
    checkpoint the reference writes -- ``<directory>/tf_ckpts/ckpt-N`` or ``<directory>/ckpt-N``
    (tf.train.Checkpoint(variables=model.variables, ...), train_utils.py:62-75; read by tf_checkpoint.py)."""
    path = os.path.join(directory, "weights.npz")
    if os.path.exists(path):
        with np.load(path) as z:
            return {k: z[k] for k in z.files}
    from . import tf_checkpoint
    for d in (os.path.join(directory, "tf_ckpts"), directory):
        prefix = tf_checkpoint.latest_checkpoint(d)
        if prefix is not None:
            return tf_checkpoint.import_variables(prefix, shapes)
    raise FileNotFoundError(f"{directory}: neither weights.npz nor a TensorFlow checkpoint (tf_ckpts/ckpt-N.index)")


def _npz_loader(root: str, shapes: Dict[str, tuple]) -> Callable[[float], Optional[Dict[str, np.ndarray]]]:
    def load(sigma: float):
        return load_weights(os.path.join(root, "sigma_" + str(round(sigma, 2))), shapes)        # run_basis_sep.py:284-285
    return load


def glow_precision(args) -> int:
    """Arithmetic of the Glow priors.  Default: the tensor-core parity mode ASEP_PREC_FP16X3 (three split-precision
    products per GEMM: log_prob, round trip, score and per-step Langevin gates of DESIGN.md section 4); ``--fast``: one
    bf16 product (3.2x the throughput; score within ~5e-2, per-step gate met on the annealed half of the schedule);
    ``--precision`` names any mode; ``--exact`` keeps its round-1 meaning (fp32 CUDA cores).  Widths other than 512
    filters have no tensor-core kernel and run on the fp32 CUDA-core path."""
    from . import _lib
    table = {"fp32": _lib.PREC_FP32, "bf16": _lib.PREC_BF16, "fp16": _lib.PREC_FP16, "bf16x2": _lib.PREC_BF16X2,
             "fp16x2": _lib.PREC_FP16X2, "fp16x3": _lib.PREC_FP16X3}
    if int(args.n_filters) != 512:
        return _lib.PREC_FP32
    name = getattr(args, "precision", None)
    if name:
        if name not in table:
            raise ValueError(f"--precision should be one of {sorted(table)}")
        return table[name]
    if getattr(args, "exact", False):
        return _lib.PREC_FP32
    return _lib.PREC_BF16 if getattr(args, "fast", False) else _lib.PREC_FP16X3


def build_models(args, sigmas, device_index: int):
    """One prior per restore directory (reference: run_basis_sep.py:386-397) and their per-sigma weight suppliers:
    (models, ckpts), both of length K."""
    from . import _lib
    from .flow_models.flow_builder import build_glow
    from .weights import init_glow_params
    restores = restore_dirs(args)
    if args.model_type == "glow":
        cfg = GlowConfig(H=args.height, W=args.width, C=1, L=args.L, K=args.K, n_filters=args.n_filters,
                         learntop=bool(args.learntop), minval=0.0, maxval=1.0)
        models, ckpts = [], []
        for i, restore in enumerate(restores):
            if args.random_init is not None:
                params = init_glow_params(cfg, seed=int(args.random_init) + i, mode="perturbed")
                ckpts.append(None)
            else:
                from .weights import glow_param_shapes
                ckpts.append(_npz_loader(os.path.abspath(restore), glow_param_shapes(cfg)))
                params = ckpts[-1](float(sigmas[0]))
            models.append(build_glow(None, [args.height, args.width, 1], L=args.L, K=args.K, n_filters=args.n_filters,
                                     learntop=args.learntop, l2_reg=args.l2_reg, data_type="melspec", minval=0.0,
                                     maxval=1.0, use_logit=False, params=params, precision=glow_precision(args)))
        return models, ckpts
    from .ncsn.utils import get_uncompiled_model, get_uncompiled_model_v2
    builders = []
    for i, restore in enumerate(restores):
        params = None
        if args.random_init is None:
            from .ncsn.utils import _ncsn_cfg
            from .weights import ncsn_param_shapes
            params = load_weights(os.path.abspath(restore), ncsn_param_shapes(_ncsn_cfg(args, args.version)))
        if args.version == "v1":
            builders.append(get_uncompiled_model(args, name=f"model{i + 1}", params=params,
                                                 seed=None if args.random_init is None else int(args.random_init) + i))
        else:
            builders.append(get_uncompiled_model_v2(args, sigmas=sigmas, name=f"model{i + 1}", params=params,
                                                    seed=None if args.random_init is None else int(args.random_init) + i))
    return builders, [None] * len(builders)


# --------------------------------------------------------------------------------------- sources
MAX_SOURCES = 8                     # the fused update keeps the state of every source in registers (csrc/langevin.cu)


def restore_dirs(args) -> List[str]:
    """The K restore directories, one prior per source: RESTORE1 RESTORE2 [RESTORE ...]."""
    dirs = [args.RESTORE1, args.RESTORE2] + list(getattr(args, "RESTORE", None) or [])
    if len(dirs) > MAX_SOURCES:
        raise ValueError(f"BASIS separates at most {MAX_SOURCES} sources; {len(dirs)} restore directories were given")
    return dirs


def source_names(args) -> List[str]:
    """Stem names of the K sources (``--sources``): ``<song_dir>/<name>.wav`` or ``.npy``.  The default piano,violin is
    the reference's two-source layout; with more sources and a song directory, --sources is required."""
    K = len(restore_dirs(args))
    spec = getattr(args, "sources", None)
    if spec is None:
        if K == 2:
            return ["piano", "violin"]
        if args.song_dir is not None and not getattr(args, "synthetic", False):
            raise ValueError(f"--sources is required to name the {K} stems in --song_dir")
        return [f"source{k + 1}" for k in range(K)]
    names = [nm.strip() for nm in spec.split(",")]
    if len(names) != K or not all(names):
        raise ValueError(f"--sources names {len(names)} stems ({spec!r}), but there are {K} restore directories")
    return names


# --------------------------------------------------------------------------------------- main
def build_parser() -> argparse.ArgumentParser:
    """The reference's flags (run_basis_sep.py:453-523) plus --synthetic / --random_init / --seed, and K sources:
    RESTORE1 RESTORE2 [RESTORE ...] with --sources."""
    p = argparse.ArgumentParser(description="BASIS Separatation")
    p.add_argument("RESTORE1", type=str, default=None, help="directory of saved model1")
    p.add_argument("RESTORE2", type=str, default=None, help="directory of saved model2")
    p.add_argument("RESTORE", type=str, nargs="*", default=[],
                   help="directories of the priors of sources 3..K (K <= 8): one prior per source")
    p.add_argument("--output", type=str, default="basis_sep")
    p.add_argument("--debug", action="store_true")
    p.add_argument("--dataset", type=str, default="melspec")
    p.add_argument("--song_dir", type=str, default=None)
    p.add_argument("--inverse", action="store_true", help="accepted; audio inversion is outside the hot path")
    p.add_argument("--model_type", type=str, default="ncsn")
    p.add_argument("--n_mixed", type=int, default=30)
    p.add_argument("--config", type=str)
    p.add_argument("--height", type=int, default=96)
    p.add_argument("--width", type=int, default=64)
    p.add_argument("--scale", type=str, default="dB")
    p.add_argument("--T", type=int, default=100)
    p.add_argument("--sigma1", type=float, default=1.0)
    p.add_argument("--sigmaL", type=float, default=0.01)
    p.add_argument("--num_classes", type=int, default=10)            # the reference parses a float (defect D7)
    p.add_argument("--progression", type=str, default="geometric")
    p.add_argument("--n_filters", type=int, default=192)
    p.add_argument("--version", type=str, default="v1")
    p.add_argument("--L", default=3, type=int)
    p.add_argument("--K", type=int, default=32)
    p.add_argument("--l2_reg", type=float, default=None)
    p.add_argument("--learntop", action="store_true")
    p.add_argument("--optimizer", type=str, default="adamax")
    p.add_argument("--batch_size", type=int, default=256)
    p.add_argument("--learning_rate", type=float, default=0.001)
    p.add_argument("--use_logit", action="store_true")
    p.add_argument("--alpha", type=float, default=10 ** (-6))
    # additions
    p.add_argument("--synthetic", action="store_true", help="separate seeded synthetic mel patches")
    p.add_argument("--random_init", type=int, default=None, metavar="SEED", help="seeded random-init weights")
    p.add_argument("--seed", type=int, default=0, help="Philox seed of the Langevin noise and of x1/x2 init")
    p.add_argument("--fast", action="store_true",
                   help="throughput mode: one bf16 tensor-core product per GEMM / convolution (default: the parity modes, "
                        "three split-precision products: Glow ASEP_PREC_FP16X3, score networks ASEP_PREC_BF16X3)")
    p.add_argument("--precision", type=str, default=None,
                   help="Glow priors: fp32 | bf16 | fp16 | bf16x2 | fp16x2 | fp16x3 (overrides --fast / --exact)")
    p.add_argument("--exact", action="store_true",
                   help="Glow priors on the fp32 CUDA-core kernels (the on-device checker); score networks: the parity mode")
    p.add_argument("--sources", type=str, default=None, metavar="NAME,...",
                   help="stem names of the K sources in --song_dir (<name>.wav or <name>.npy); default piano,violin (K = 2)")
    p.add_argument("--host_loop", action="store_true",
                   help="run the sigma loop on the host (one library call per noise level) instead of asep_basis_*_run")
    p.add_argument("--mix", type=str, default=None, metavar="PATH",
                   help="separate this whole wav file from the mixture alone (no stems needed): overlapping 2.04 s segments, "
                        "<output>/<source name>.wav per source at the input's rate and length; --n_mixed is ignored")
    p.add_argument("--overlap_frames", type=int, default=8,
                   help="with --mix: STFT frames (512 samples at 16 kHz) two neighbouring segments share and cross-fade "
                        "over, 0..31 (0: hard cuts)")
    p.add_argument("--wiener_filter", action="store_true",
                   help="with --mix: invert through the K-source Wiener filter instead of the mixture's phase")
    p.add_argument("--render", choices=("mel", "mask"), default="mel",
                   help="with --mix: how the stems are made from the separated mel spectrograms.  mel (default): inverted at "
                        "16 kHz (mono, 133 Hz .. 7.6 kHz) and resampled; mask: multichannel Wiener masks applied to the "
                        "recording itself (its channels, rate and full band; the stems sum to it)")
    p.add_argument("--mwf_iterations", type=int, default=None, metavar="N",
                   help="with --render mask: EM iterations of the multichannel Wiener filter, 0..10 (default 1)")
    return p


def check_mix_args(args) -> None:
    """Flag rules of the whole-track mode (--mix), checked before anything runs on the device: no --song_dir / --synthetic
    next to it, --overlap_frames in 0..31, --sources (if given) naming one output per restore directory, and --render mask
    only with --mix, without --wiener_filter, with --mwf_iterations in 0..10 (which belongs to --render mask alone)."""
    render = getattr(args, "render", "mel")
    iterations = getattr(args, "mwf_iterations", None)
    if render == "mask":
        if getattr(args, "mix", None) is None:
            raise ValueError("--render mask renders a whole recording: it needs --mix")
        if args.wiener_filter:
            raise ValueError("--render mask is a multichannel Wiener filter of its own; --wiener_filter does not apply")
        if iterations is not None:
            from .track import check_mwf_iterations
            check_mwf_iterations(iterations)
    elif iterations is not None:
        raise ValueError("--mwf_iterations belongs to --render mask")
    if getattr(args, "mix", None) is None:
        return
    if args.song_dir is not None or getattr(args, "synthetic", False):
        raise ValueError("--mix separates a mixture on its own; it cannot be combined with --song_dir or --synthetic")
    from .track import check_overlap_frames
    check_overlap_frames(args.overlap_frames)
    source_names(args)


def merge_config(args: argparse.Namespace) -> argparse.Namespace:
    """YAML over argparse defaults, CLI-only fields preserved (fixes defect D2; reference :269-278)."""
    if args.config is None:
        return args
    cfg = vars(get_config(args.config))
    keep = ("dataset", "debug", "output", "song_dir", "inverse", "model_type", "n_mixed", "RESTORE1", "RESTORE2",
            "synthetic", "random_init", "seed", "config", "fast", "precision", "exact", "host_loop", "RESTORE", "sources", "mix",
            "overlap_frames", "wiener_filter", "render", "mwf_iterations")
    merged = dict(vars(args))
    for k, v in cfg.items():
        if k not in keep:
            merged[k] = v
    merged["num_classes"] = int(merged["num_classes"])
    return argparse.Namespace(**merged)


def main(args) -> Optional[Dict[str, np.ndarray]]:
    import torch
    import torch.distributed as dist

    from . import track
    args = merge_config(args)
    check_mix_args(args)
    mix_mode = getattr(args, "mix", None) is not None
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("run_basis_sep needs a CUDA (sm_100a) device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)

    sigmas = get_sigmas(args.sigma1, args.sigmaL, args.num_classes, progression=args.progression)
    if args.model_type not in ("glow", "ncsn"):
        raise ValueError("model_type should be 'ncsn' or 'glow'")
    args.data_shape = [args.height, args.width, 1]
    args.data_type = "melspec"
    if args.scale == "dB":
        args.maxval, args.minval = 20.0, -100.0
    elif args.scale == "power":
        raise NotImplementedError("the power-scale mixing is not used by configs/melspec_*.yml")
    else:
        raise ValueError("scale should be 'power' or 'dB'")

    out_dir = os.path.abspath(args.output)
    os.makedirs(out_dir, exist_ok=True)
    log_file = None
    old_stdout = sys.stdout
    if rank == 0 and not args.debug:
        log_file = open(os.path.join(out_dir, "out.log"), "w")
        sys.stdout = log_file
    elif rank != 0:
        sys.stdout = open(os.devnull, "w")
    try:
        t0 = time.time()
        if mix_mode:
            mask = getattr(args, "render", "mel") == "mask"
            audio = track.read_track_channels(os.path.abspath(args.mix)) if mask else None     # > 2 channels fail here
            mix_db, stft_mixture, seg = load_mix_patches(args)
            gts, K = None, len(restore_dirs(args))
        else:
            mix_db, gts, stft_mixture = load_song_patches(args)
            K = len(gts)
        n = mix_db.shape[0]
        lo, hi = shard_range(n, world, rank)
        mixed_full = ((mix_db - args.minval) / (args.maxval - args.minval)).astype(np.float32)   # :355
        rng = np.random.Generator(np.random.PCG64(args.seed))
        x_full = np.stack([rng.uniform(0.0, 1.0, mixed_full.shape).astype(np.float32) for _ in range(K)])   # :360-361
        mixed = torch.as_tensor(mixed_full[lo:hi]).to(dev)
        x = torch.as_tensor(np.ascontiguousarray(x_full[:, lo:hi])).to(dev)
        args.elem_offset = lo * args.height * args.width
        print("Data Loaded in {} seconds".format(round(time.time() - t0, 3)))
        post_processing = post_processing_fn(args)
        models, ckpts = build_models(args, sigmas, local_rank)
        template = "BASIS Separation \n\t "
        for k, v in vars(args).items():
            template += "{} = {} \n\t ".format(k, v)
        print(template)
        torch.cuda.synchronize()
        t0 = time.time()
        if hi > lo:
            x, x_arr = basis_outer_loop_k(mixed, x, models, None, sigmas, ckpts, args, None)
        else:
            x_arr = {f"x{k + 1}": [x[k].cpu().numpy()] * (len(sigmas) + 1) for k in range(K)}
        torch.cuda.synchronize()
        t1 = time.time()
        print("Duration: {} seconds".format(round(t1 - t0, 3)))
        # final gather: the only cross-GPU traffic (SURVEY.md 8(e))
        x_all = [gather_segments(x[k].cpu().numpy(), n) for k in range(K)]
        conv = [gather_segments(np.array(x_arr[f"x{k + 1}"]), n, axis=1) for k in range(K)]
        results = None
        if rank == 0:
            if mix_mode:
                results = track.track_results([post_processing(x_all[k].squeeze(-1)) for k in range(K)],
                                              post_processing(mixed_full.squeeze(-1)), stft_mixture, seg["starts"],
                                              seg["track_length"], seg["orig_sr"], seg["orig_length"], args.overlap_frames)
            else:
                results = {f"x{k + 1}": post_processing(x_all[k].squeeze(-1)) for k in range(K)}
                results.update({f"gt{k + 1}": gts[k].squeeze(-1) for k in range(K)})
                results.update({"mixed": post_processing(mixed_full.squeeze(-1)), "stft_mixture": stft_mixture})
            np.savez(os.path.join(out_dir, "results"), **results)                                # :435
            np.savez(os.path.join(out_dir, "results_convergence"),
                     **{f"x{k + 1}": post_processing(conv[k]) for k in range(K)})
            if mix_mode:                                                 # whole-track back end: one wav per source
                t2 = time.time()
                if mask:
                    n_iter = 1 if args.mwf_iterations is None else args.mwf_iterations
                    tracks = track.render_results(results, os.path.abspath(args.mix), n_iter, audio)
                else:
                    tracks = track.invert_results(results, args.wiener_filter)
                names = source_names(args)
                track.write_tracks(out_dir, names, tracks, seg["orig_sr"])
                print("Inversion duration: {} seconds".format(round(time.time() - t2, 3)))
                results["separated"] = dict(zip(names, tracks))
            results["duration_s"] = t1 - t0
        return results
    finally:
        if sys.stdout is not old_stdout:
            try:
                sys.stdout.close()
            except Exception:
                pass
        sys.stdout = old_stdout


def cli(argv=None):
    return main(build_parser().parse_args(argv))


if __name__ == "__main__":
    cli()
