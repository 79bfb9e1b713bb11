"""Functional access to the stateless kernels of libasep.so (single bijectors, Langevin update)."""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib


def _prep(t: torch.Tensor) -> torch.Tensor:
    dev = torch.device("cuda", _lib.init())
    if t.dtype != torch.float32:
        t = t.float()
    return t.to(dev).contiguous()


def actnorm(x, log_scale, shift, inverse: bool = False) -> torch.Tensor:
    """ActNorm._forward / _inverse (reference: flow_tfp_bijectors.py:242-247)."""
    x, log_scale, shift = _prep(x), _prep(log_scale), _prep(shift)
    y = torch.empty_like(x)
    a, b, c, d = _lib.dl(x), _lib.dl(log_scale), _lib.dl(shift), _lib.dl(y)
    _lib.check(_lib.load().asep_actnorm(a.ptr, b.ptr, c.ptr, d.ptr, int(inverse), _lib.stream_ptr()))
    return y


def inv1x1(x, w) -> torch.Tensor:
    """y[..., o] = sum_i x[..., i] w[i, o]  (reference: flow_tfp_bijectors.py:304-305, :316)."""
    x, w = _prep(x), _prep(w)
    y = torch.empty_like(x)
    a, b, c = _lib.dl(x), _lib.dl(w), _lib.dl(y)
    _lib.check(_lib.load().asep_inv1x1(a.ptr, b.ptr, c.ptr, _lib.stream_ptr()))
    return y


def coupling(x, r, inverse: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """AffineCouplingLayerSplit given r = [raw_log_s | t]; returns (y, log-det of this direction)."""
    x, r = _prep(x), _prep(r)
    y = torch.empty_like(x)
    ld = torch.empty((x.shape[0],), dtype=torch.float32, device=x.device)
    a, b, c, d = _lib.dl(x), _lib.dl(r), _lib.dl(y), _lib.dl(ld)
    _lib.check(_lib.load().asep_coupling(a.ptr, b.ptr, c.ptr, d.ptr, int(inverse), _lib.stream_ptr()))
    return y, ld


def squeeze(x, inverse: bool = False) -> torch.Tensor:
    """Squeeze._forward / _inverse (reference: flow_tfp_bijectors.py:170-180)."""
    x = _prep(x)
    N, H, W, C = x.shape
    if not inverse:
        if H % 2 or W % 2:
            raise ValueError("Squeeze needs even H and W")
        y = torch.empty((N, H // 2, W // 2, 4 * C), dtype=torch.float32, device=x.device)
    else:
        if C % 4:
            raise ValueError("inverse Squeeze needs C divisible by 4")
        y = torch.empty((N, H * 2, W * 2, C // 4), dtype=torch.float32, device=x.device)
    a, b = _lib.dl(x), _lib.dl(y)
    _lib.check(_lib.load().asep_squeeze(a.ptr, b.ptr, int(inverse), _lib.stream_ptr()))
    return y


# ---- two sources: the K = 2 case of the stacked calls below, for callers that hold x1 and x2 as separate tensors
def _pair(x1, x2) -> torch.Tensor:
    """The stacked [2, ...] state of ``x1, x2``; the calls copy it back into them (they are updated in place)."""
    for t in (x1, x2):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise ValueError("x1/x2 must be contiguous float32 CUDA tensors (updated in place)")
    if x1.shape != x2.shape:
        raise ValueError(f"x1 {tuple(x1.shape)} and x2 {tuple(x2.shape)} must have the same shape")
    return torch.stack([x1, x2])


def _unpair(x, x1, x2) -> None:
    x1.copy_(x[0])
    x2.copy_(x[1])


def _noise_pair(n1, n2, dim: int) -> Optional[torch.Tensor]:
    """The injected draws of both sources stacked on the source axis ``dim``, or None for in-kernel Philox noise."""
    if (n1 is None) != (n2 is None):
        raise ValueError("inject both noise tensors or neither")
    return None if n1 is None else torch.stack([_prep(n1), _prep(n2)], dim)


def mixing_db(x1, x2):
    """g(x1,x2) and grad_g (reference: run_basis_sep.py:131-147)."""
    g, w = mixing_db_k(torch.stack([_prep(x1), _prep(x2)]))
    return g, w[0], w[1]


def langevin_step(x1, x2, s1, s2, mixed, eta: float, lam: float, noise_scale: float,
                  n1: Optional[torch.Tensor] = None, n2: Optional[torch.Tensor] = None, seed: int = 0,
                  step: int = 0, elem_offset: int = 0, nan_count: Optional[torch.Tensor] = None) -> None:
    """In-place fused update of both sources (reference: run_basis_sep.py:163-181)."""
    noise, x = _noise_pair(n1, n2, 0), _pair(x1, x2)
    langevin_step_k(x, torch.stack([_prep(s1), _prep(s2)]), mixed, eta, lam, noise_scale, noise=noise, seed=seed, step=step,
                    elem_offset=elem_offset, nan_count=nan_count)
    _unpair(x, x1, x2)


def philox_normal(shape, seed: int, step: int, stream_id: int, elem_offset: int = 0) -> torch.Tensor:
    dev = torch.device("cuda", _lib.init())
    out = torch.empty(shape, dtype=torch.float32, device=dev)
    d = _lib.dl(out)
    _lib.check(_lib.load().asep_philox_normal(d.ptr, int(seed), int(step), int(stream_id), int(elem_offset),
                                              _lib.stream_ptr()))
    return out


def basis_glow_inner(m1, m2, mixed, x1, x2, T: int, eta: float, lam: float, noise_scale: float,
                     noise1=None, noise2=None, seed: int = 0, step0: int = 0, elem_offset: int = 0,
                     per_step: Optional[torch.Tensor] = None, nan_count: Optional[torch.Tensor] = None) -> None:
    """T Langevin steps at one noise level with two Glow priors, entirely inside the library.  ``noise1/noise2``: [T, ...]
    each; ``per_step``: [T, 2, ...]."""
    noise, x = _noise_pair(noise1, noise2, 1), _pair(x1, x2)
    basis_glow_inner_k([m1, m2], mixed, x, T, eta, lam, noise_scale, noise=noise, seed=seed, step0=step0,
                       elem_offset=elem_offset, per_step=per_step, nan_count=nan_count)
    _unpair(x, x1, x2)


def basis_ncsn_inner(m1, m2, mixed, x1, x2, sigma_idx: int, T: int, eta: float, lam: float, noise_scale: float,
                     noise1=None, noise2=None, seed: int = 0, step0: int = 0, elem_offset: int = 0,
                     per_step: Optional[torch.Tensor] = None, nan_count: Optional[torch.Tensor] = None) -> None:
    """T Langevin steps at noise level ``sigma_idx`` with two NCSN score networks, inside the library (arguments as
    basis_glow_inner)."""
    noise, x = _noise_pair(noise1, noise2, 1), _pair(x1, x2)
    basis_ncsn_inner_k([m1, m2], mixed, x, sigma_idx, T, eta, lam, noise_scale, noise=noise, seed=seed, step0=step0,
                       elem_offset=elem_offset, per_step=per_step, nan_count=nan_count)
    _unpair(x, x1, x2)


def basis_run(m1, m2, mixed, x1, x2, T: int, eta, lam, noise_scale, seed: int = 0, elem_offset: int = 0,
              snapshots: Optional[torch.Tensor] = None, nan_count: Optional[torch.Tensor] = None) -> None:
    """The whole sigma x T loop inside the library (reference: run_basis_sep.py:217-260): ``eta / lam / noise_scale`` are
    length-L sequences of the per-level float32 constants.  ``m1 / m2``: two score networks, two Glow priors, or two
    length-L lists of Glow priors (one fine-tuned pair per noise level); ``snapshots``: None or [L, 2, ...]."""
    x = _pair(x1, x2)
    models = [[a, b] for a, b in zip(m1, m2, strict=True)] if isinstance(m1, (list, tuple)) else [m1, m2]
    basis_run_k(models, mixed, x, T, eta, lam, noise_scale, seed=seed, elem_offset=elem_offset, snapshots=snapshots,
                nan_count=nan_count)
    _unpair(x, x1, x2)


# ---- K sources (2 <= K <= 8): stacked [K, ...] states, [T, K, ...] noise / per-step dumps, [L, K, ...] snapshots
def _state_k(x) -> None:
    if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()):
        raise ValueError("x must be a contiguous float32 CUDA tensor [K, ...] (updated in place)")


def _handles(models):
    import ctypes
    return (ctypes.c_void_p * len(models))(*[m.handle.value for m in models])


def mixing_db_k(x):
    """g(x_1..x_K) and grad_g = softmax_k of a stacked ``x`` [K, ...] (reference: run_basis_sep.py:106-149)."""
    x = _prep(x)
    g, w = torch.empty_like(x[0]), torch.empty_like(x)
    t = [_lib.dl(v) for v in (x, g, w)]
    _lib.check(_lib.load().asep_mixing_db_k(int(x.shape[0]), *(v.ptr for v in t), _lib.stream_ptr()))
    return g, w


def langevin_step_k(x, score, mixed, eta: float, lam: float, noise_scale: float, noise: Optional[torch.Tensor] = None,
                    seed: int = 0, step: int = 0, elem_offset: int = 0, nan_count: Optional[torch.Tensor] = None) -> None:
    """In-place fused update of all K sources of ``x`` [K, ...] (reference: run_basis_sep.py:163-181); ``noise``: NULL
    (Philox, source k on stream k + 1) or [K, ...] standard normals."""
    _state_k(x)
    score, mixed = _prep(score), _prep(mixed)
    noise = None if noise is None else _prep(noise)
    t = [_lib.dl(v) for v in (x, score, mixed, noise, nan_count)]
    _lib.check(_lib.load().asep_langevin_step_k(int(x.shape[0]), t[0].ptr, t[1].ptr, t[2].ptr, t[3].ptr, float(eta),
                                                float(lam), float(noise_scale), int(seed), int(step), int(elem_offset),
                                                t[4].ptr, _lib.stream_ptr()))


def basis_glow_inner_k(models, mixed, x, T: int, eta: float, lam: float, noise_scale: float, noise=None, seed: int = 0,
                       step0: int = 0, elem_offset: int = 0, per_step: Optional[torch.Tensor] = None,
                       nan_count: Optional[torch.Tensor] = None) -> None:
    """T Langevin steps at one noise level with K Glow priors (``models[k]`` for source k of ``x`` [K, ...])."""
    _state_k(x)
    mixed = _prep(mixed)
    noise = None if noise is None else _prep(noise)
    t = [_lib.dl(v) for v in (mixed, x, noise, per_step, nan_count)]
    _lib.check(_lib.load().asep_basis_glow_inner_k(len(models), _handles(models), t[0].ptr, t[1].ptr, int(T), float(eta),
                                                   float(lam), float(noise_scale), t[2].ptr, int(seed), int(step0),
                                                   int(elem_offset), t[3].ptr, t[4].ptr, _lib.stream_ptr()))


def basis_ncsn_inner_k(models, mixed, x, sigma_idx: int, T: int, eta: float, lam: float, noise_scale: float, noise=None,
                       seed: int = 0, step0: int = 0, elem_offset: int = 0, per_step: Optional[torch.Tensor] = None,
                       nan_count: Optional[torch.Tensor] = None) -> None:
    """T Langevin steps at noise level ``sigma_idx`` with K score networks (``models[k]`` for source k of ``x``)."""
    _state_k(x)
    mixed = _prep(mixed)
    noise = None if noise is None else _prep(noise)
    t = [_lib.dl(v) for v in (mixed, x, noise, per_step, nan_count)]
    _lib.check(_lib.load().asep_basis_ncsn_inner_k(len(models), _handles(models), t[0].ptr, t[1].ptr, int(sigma_idx),
                                                   int(T), float(eta), float(lam), float(noise_scale), t[2].ptr, int(seed),
                                                   int(step0), int(elem_offset), t[3].ptr, t[4].ptr, _lib.stream_ptr()))


def basis_run_k(models, mixed, x, T: int, eta, lam, noise_scale, seed: int = 0, elem_offset: int = 0,
                snapshots: Optional[torch.Tensor] = None, nan_count: Optional[torch.Tensor] = None) -> None:
    """The whole sigma x T loop over K sources inside the library (reference: run_basis_sep.py:217-260).  ``models``: K
    score networks, K Glow priors, or L lists of K Glow priors (one fine-tuned set per noise level); ``snapshots``:
    NULL or [L, K, ...]."""
    import ctypes
    _state_k(x)
    L = len(eta)
    arr = [(ctypes.c_float * L)(*[float(v) for v in seq]) for seq in (eta, lam, noise_scale)]
    mixed = _prep(mixed)
    t = [_lib.dl(v) for v in (mixed, x, snapshots, nan_count)]
    per_level = isinstance(models[0], (list, tuple))
    first = models[0][0] if per_level else models[0]
    if hasattr(first, "cfg") and hasattr(first.cfg, "K"):                 # Glow priors
        sets = [list(s) for s in models] if per_level else [list(models)]
        K = len(sets[0])
        if any(len(s) != K for s in sets):
            raise ValueError("every noise level needs the same number of priors")
        flat = [m for s in sets for m in s]
        _lib.check(_lib.load().asep_basis_glow_run_k(K, _handles(flat), len(sets), t[0].ptr, t[1].ptr, L, int(T), arr[0],
                                                     arr[1], arr[2], int(seed), int(elem_offset), t[2].ptr, t[3].ptr,
                                                     _lib.stream_ptr()))
    else:
        if per_level:
            raise ValueError("per-level model lists are a Glow feature; score networks are conditioned on the level")
        _lib.check(_lib.load().asep_basis_ncsn_run_k(len(models), _handles(models), t[0].ptr, t[1].ptr, L, int(T), arr[0],
                                                     arr[1], arr[2], int(seed), int(elem_offset), t[2].ptr, t[3].ptr,
                                                     _lib.stream_ptr()))


# ---- the tcgen05 convolutions of the score networks one launch at a time (tests compare each with a float64 reference)
def _bf16(t: torch.Tensor, what: str) -> torch.Tensor:
    if t.dtype != torch.bfloat16:
        raise ValueError(f"{what} must be a bfloat16 tensor (got {t.dtype})")
    return t.to(torch.device("cuda", _lib.init())).contiguous()


def conv_tc_image(kernel, transposed: bool = False, lo: bool = False, on_device: bool = True) -> torch.Tensor:
    """bf16 SWIZZLE_128B tile image [k*k*Cin*Cout] of the HWIO fp32 ``kernel`` as the device builder of the training step
    (``on_device``) or the host builder of ``asep_ncsn_prepare`` makes it; ``transposed``: the data-gradient image,
    ``lo``: the low word of the split-bf16 pair."""
    k = torch.as_tensor(kernel)
    k = _prep(k) if on_device else k.float().contiguous()
    img = torch.empty(k.numel(), dtype=torch.bfloat16, device=torch.device("cuda", _lib.init()))
    a, b = _lib.dl(k), _lib.dl(img)
    _lib.check(_lib.load().asep_conv_tc_image(a.ptr, int(transposed), int(lo), int(on_device), b.ptr, _lib.stream_ptr()))
    return img


def conv_tc_forward(img, x, ksize: int, cin: int, cout: int, dil: int = 1, bias=None, add=None, add2=None, out=None,
                    stats: bool = False, out_bf16: bool = False):
    """One ``k_conv_tc`` / ``k_conv_tc_sw`` launch: ``out`` [N,H,W,cout] fp32 = conv(x bf16 [N,H,W,cin]) + bias + add +
    add2.  ``out`` may be passed (and be ``add``: the split-bf16 passes accumulate in place).  Returns (out, stats
    [N,cout,2] float64 or None, bf16 copy of out or None)."""
    img, x = _bf16(img, "img"), _bf16(x, "x")
    if out is None:
        out = torch.empty(tuple(x.shape[:3]) + (cout,), dtype=torch.float32, device=x.device)
    elif not (out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()):
        raise ValueError("out must be a contiguous float32 CUDA tensor")
    bias = None if bias is None else _prep(bias)
    if add is not None and add is not out:
        add = _prep(add)
    add2 = None if add2 is None else _prep(add2)
    st = torch.empty((x.shape[0], cout, 2), dtype=torch.float64, device=x.device) if stats else None
    ob = torch.empty(tuple(x.shape[:3]) + (cout,), dtype=torch.bfloat16, device=x.device) if out_bf16 else None
    t = [_lib.dl(v) for v in (img, bias, x, add, add2, out, st, ob)]
    _lib.check(_lib.load().asep_conv_tc_forward(t[0].ptr, t[1].ptr, int(ksize), int(cin), int(cout), int(dil), t[2].ptr,
                                                t[3].ptr, t[4].ptr, t[5].ptr, t[6].ptr, t[7].ptr, _lib.stream_ptr()))
    return out, st, ob


def conv_wgrad_tc(x, g, dk: torch.Tensor, ksize: int, dil: int = 1) -> torch.Tensor:
    """One ``k_conv_wgrad_tc`` launch: ``dk`` fp32 [k,k,Cin,Cout] (a contiguous CUDA tensor, updated in place) += the
    weight gradient of the 'same' convolution for input x bf16 [N,H,W,Cin] and output gradient g bf16 [N,H,W,Cout]."""
    x, g = _bf16(x, "x"), _bf16(g, "g")
    if not (dk.is_cuda and dk.dtype == torch.float32 and dk.is_contiguous()):
        raise ValueError("dk must be a contiguous float32 CUDA tensor (it is accumulated into)")
    t = [_lib.dl(v) for v in (x, g, dk)]
    _lib.check(_lib.load().asep_conv_wgrad_tc(t[0].ptr, t[1].ptr, t[2].ptr, int(ksize), int(dil), _lib.stream_ptr()))
    return dk


# ---- the tcgen05 coupling network of the Glow prior one launch at a time (tests compare each with a float64 reference)
def glow_coupling_tc(glow, block: int, step: int, backward: bool, src, G, mask1=None, mask2=None, dump1=None, dump2=None,
                     out=None) -> None:
    """One ``k_nn_tc4`` / ``k_nn_tcx`` launch with the prepared weights of (block, step) of ``glow`` (a ``Glow`` in a
    tensor-core precision), on caller tensors that are passed as they are: the library checks every one before the
    launch (layouts in include/asep.h).  src fp32 [N,Hb,Wb,Cb]; G fp32 [nparts, ceil(M/128)*128*n3p]; mask1 / mask2 int32
    [M,16] (outputs of the forward, inputs of the backward); dump1 / dump2 bf16 [M,512]; out fp32 r [N,Hb,Wb,Cb] or gxb
    [N,Hb,Wb,Cb/2]."""
    t = [_lib.dl(v) for v in (src, mask1, mask2, dump1, dump2, G, out)]
    _lib.check(_lib.load().asep_glow_coupling_tc(glow.handle, int(block), int(step), int(backward), t[0].ptr, t[1].ptr,
                                                 t[2].ptr, t[3].ptr, t[4].ptr, t[5].ptr, t[6].ptr, _lib.stream_ptr()))


def glow_wgrad_tc(A, B, n_valid: int, out) -> None:
    """One ``k_wgrad_tc`` launch: ``out`` fp32 [512, ldo] += A^T B for the columns < n_valid, A bf16 [P,512], B bf16
    [P,ldb] (passed as they are; the library checks them)."""
    t = [_lib.dl(v) for v in (A, B, out)]
    _lib.check(_lib.load().asep_glow_wgrad_tc(t[0].ptr, t[1].ptr, int(n_valid), t[2].ptr, _lib.stream_ptr()))
