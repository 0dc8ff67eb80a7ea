"""Shared test helpers (no CUDA needed to import)."""
import os
import re

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class ReplayNoise:
    """Noise source for the PRODUCT filter (protocol of multimodalfilter_b200.torchfilter.filters):
    replays pre-drawn CPU tensors, moving them to the filter's device."""

    def __init__(self, *, init_eps=None, process_eps=(), uniforms=()):
        self._init, self._eps, self._u = init_eps, list(process_eps), list(uniforms)

    def init_eps(self, M, N, sd, like):
        assert self._init.shape == (M, N, sd)
        return self._init

    def process_eps(self, rows, sd, like):
        eps = self._eps.pop(0)
        assert eps.shape == (rows, sd)
        return eps

    def resample_uniforms(self, N, S, like):
        return self._u.pop(0)

    def randperm(self, M):
        return torch.randperm(M)


def draw_noise(T, N, M, sd, seed, systematic=False):
    g = torch.Generator().manual_seed(seed)
    init = torch.randn(M, N, sd, generator=g)
    eps = [torch.randn(N * M, sd, generator=g) for _ in range(T)]
    if systematic:
        us = [torch.rand(N, dtype=torch.float64, generator=g) for _ in range(T)]
    else:
        us = [torch.rand(N * M, dtype=torch.float64, generator=g).reshape(N, M) for _ in range(T)]
    return init, eps, us


def assert_close(actual, expected, rtol=1e-4, atol=None, msg=""):
    """|a - e| <= rtol * max(|e|, scale) with scale = the RMS of the expected tensor: the north
    star's "1e-4 relative in fp32", made robust to entries that happen to be near zero."""
    a = np.asarray(actual, dtype=np.float64)
    e = np.asarray(expected, dtype=np.float64)
    assert a.shape == e.shape, f"{msg}: shape {a.shape} vs {e.shape}"
    finite = np.isfinite(e)
    assert np.array_equal(np.isfinite(a), finite), f"{msg}: non-finite pattern differs"
    assert np.array_equal(a[~finite], e[~finite], equal_nan=True), f"{msg}: inf/nan entries differ"
    if not finite.any():
        return
    scale = np.sqrt(np.mean(e[finite] ** 2))
    bound = rtol * np.maximum(np.abs(e), scale) + (atol or 0.0)
    err = np.abs(a - e)
    bad = finite & (err > bound)
    assert not bad.any(), (
        f"{msg}: {bad.sum()}/{bad.size} entries out of tolerance; worst |err|={err[finite].max():.3e} "
        f"(bound there {bound.reshape(-1)[np.argmax(np.where(finite, err, 0))]:.3e}, scale {scale:.3e})"
    )


def kernel_ran(names, want):
    """`want` is a kernel as the profiler demangles it, e.g. k_normalize_resample<false,32> (spaces ignored); the mangled
    spelling (k_normalize_resampleILb0ELi32EE) is accepted too."""
    base, _, args = want.partition("<")
    mangled = base
    if args:
        code = {"false": "Lb0E", "true": "Lb1E"}
        mangled += "I" + "".join(code.get(a, f"Li{a}E") for a in args.rstrip(">").split(",")) + "E"
    return any(want in n.replace(" ", "") or mangled in n for n in names)


def header_symbols():
    text = open(os.path.join(REPO, "include", "mmf_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mmf_[a-z0-9_]+)\s*\(", text)))


# ---- numpy interpreter of the packed layouts documented in include/mmf_b200.h ----------------------
U = 64


def _take(buf, pos, n):
    return buf[pos : pos + n], pos + n


def run_packed_chain(w, spec, x, rowbias):
    """w: flat fp32 pack; spec: (in_dim, n_pre, mid_relu, n_post, out_dim); x (B, in_dim); rowbias (B, 64)."""
    in_dim, n_pre, mid_relu, n_post, out_dim = spec
    pos = 0
    Wt, pos = _take(w, pos, in_dim * U)
    b, pos = _take(w, pos, U)
    h = np.maximum(x @ Wt.reshape(in_dim, U) + b, 0)

    def res(h, pos):
        W1t, pos = _take(w, pos, U * U)
        b1, pos = _take(w, pos, U)
        W2t, pos = _take(w, pos, U * U)
        b2, pos = _take(w, pos, U)
        t = np.maximum(h @ W1t.reshape(U, U) + b1, 0)
        return np.maximum(t @ W2t.reshape(U, U) + b2 + h, 0), pos

    for _ in range(n_pre):
        h, pos = res(h, pos)
    Wt, pos = _take(w, pos, U * U)
    h = h @ Wt.reshape(U, U) + rowbias
    if mid_relu:
        h = np.maximum(h, 0)
    for _ in range(n_post):
        h, pos = res(h, pos)
    W, pos = _take(w, pos, out_dim * U)
    b, pos = _take(w, pos, out_dim)
    assert pos == len(w), (pos, len(w))
    return h @ W.reshape(out_dim, U).T + b


def run_packed_rows(w, in_dim, has_encoder, u):
    pos = 0
    feats = u
    if has_encoder:
        Wt, pos = _take(w, pos, in_dim * U)
        b, pos = _take(w, pos, U)
        h = np.maximum(u @ Wt.reshape(in_dim, U) + b, 0)
        W1t, pos = _take(w, pos, U * U)
        b1, pos = _take(w, pos, U)
        W2t, pos = _take(w, pos, U * U)
        b2, pos = _take(w, pos, U)
        t = np.maximum(h @ W1t.reshape(U, U) + b1, 0)
        feats = np.maximum(t @ W2t.reshape(U, U) + b2 + h, 0)
    fd = feats.shape[1]
    Wt, pos = _take(w, pos, fd * U)
    b, pos = _take(w, pos, U)
    assert pos == len(w)
    return feats @ Wt.reshape(fd, U) + b
