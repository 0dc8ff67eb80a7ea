"""Tensor-level wrappers over the C ABI (``_lib``): shape checks, output allocation, pointer
marshalling.  Every function here launches hand-written sm_100a kernels; none has a torch or CPU
fallback."""
import ctypes as C
import os
import math

import torch

from . import _lib
from ._lib import (  # noqa: F401  (re-exported constants)
    ESTIMATE_ARGMAX,
    ESTIMATE_WEIGHTED_AVERAGE,
    PREC_BF16,
    PREC_BF16X3,
    PREC_FP32,
    RESAMPLE_MULTINOMIAL_FAST,
    RESAMPLE_MULTINOMIAL_STRICT,
    RESAMPLE_NONE,
    RESAMPLE_SYSTEMATIC_FAST,
    RESAMPLE_SYSTEMATIC_STRICT,
)

RESAMPLE_MODES = {
    "multinomial": RESAMPLE_MULTINOMIAL_STRICT,
    "multinomial_fast": RESAMPLE_MULTINOMIAL_FAST,
    "systematic": RESAMPLE_SYSTEMATIC_STRICT,
    "systematic_fast": RESAMPLE_SYSTEMATIC_FAST,
}
PRECISIONS = {"fp32": PREC_FP32, "bf16x3": PREC_BF16X3, "bf16": PREC_BF16}
ESTIMATION = {"weighted_average": ESTIMATE_WEIGHTED_AVERAGE, "argmax": ESTIMATE_ARGMAX}


class _Profile:
    """Launch counter + optional per-entry-point CUDA-event timing (events are recorded on the
    stream the kernels are launched on, i.e. torch's current stream).  Used by bench.py."""

    def __init__(self):
        self.enabled = False
        self.launches = 0
        self._events = {}

    def reset(self, enabled=False):
        self.enabled = enabled
        self.launches = 0
        self._events = {}

    def run(self, name, kernels, fn, *args):
        self.launches += kernels
        if not self.enabled:
            return _lib.call(fn, *args)
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        rc = _lib.call(fn, *args)
        stop.record()
        self._events.setdefault(name, []).append((start, stop))
        return rc

    def collect(self):
        torch.cuda.synchronize()
        kernels = {}
        for name, pairs in self._events.items():
            ms = [a.elapsed_time(b) for a, b in pairs]
            kernels[name] = {"count": len(ms), "total_ms": sum(ms), "avg_ms": sum(ms) / len(ms)}
        return {"launches": self.launches, "kernels": kernels}


PROFILE = _Profile()


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        raise _lib.MMFError(f"expected float32, got {t.dtype}")
    return t.contiguous()


def is_systematic(mode: int) -> bool:
    return mode in (RESAMPLE_SYSTEMATIC_STRICT, RESAMPLE_SYSTEMATIC_FAST)


def pack_chain_mma(chain_struct, device):
    """Build the tensor-core operand image of a chain in place: allocates the buffer, runs the pack
    kernel, stores the pointer in ``chain_struct.w_mma`` and returns the buffer (keep it alive)."""
    lib = _lib.load()
    nbytes = lib.mmf_chain_mma_bytes(C.byref(chain_struct))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
    _lib.check(_lib.call(lib.mmf_pack_chain_mma, C.byref(chain_struct), _lib.ptr(buf), _lib.stream_of(buf)))
    chain_struct.w_mma = buf.data_ptr()
    return buf


def pack_chain_bwd(chain_struct, device):
    """Backward operand image of a chain (training); stores the pointer in ``chain_struct.w_bwd``."""
    lib = _lib.load()
    nbytes = lib.mmf_chain_bwd_bytes(C.byref(chain_struct))
    buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
    _lib.check(_lib.call(lib.mmf_pack_chain_bwd, C.byref(chain_struct), _lib.ptr(buf), _lib.stream_of(buf)))
    chain_struct.w_bwd = buf.data_ptr()
    return buf


def head_depth(model_struct):
    h = model_struct.heads[0]
    return 2 * h.n_pre_res + 1 + 2 * h.n_post_res


def pf_heads_forward_train(model_struct, states, eps, rowbias, enabled_mask, precision=PREC_BF16X3):
    """Training forward of one step: move the particles (dynamics, frozen) and evaluate the heads, saving the
    activations the backward needs.  states (N,M,sd), eps (N*M,sd), rowbias (1+K,N,64) ->
    moved (N,M,sd), ll (K,N,M), act (K,L+1,16,N*M,4): chunk-major planes, act[k,l,c,p,:] = columns 4c..4c+3 of row p
    (coalesced for thread-per-row kernels; ``rows_view`` gives the (.., N*M, 64) matrix)."""
    lib = _lib.load()
    N, M, sd = states.shape
    K, L = model_struct.num_heads, head_depth(model_struct)
    states, eps, rowbias = _f32c(states), _f32c(eps), _f32c(rowbias)
    assert rowbias.shape == (1 + K, N, _lib.UNITS), f"rowbias {tuple(rowbias.shape)} != {(1 + K, N, _lib.UNITS)}"
    assert eps.numel() == N * M * sd
    dev = states.device
    moved = torch.empty_like(states)
    ll = torch.full((K, N, M), float("nan"), device=dev, dtype=torch.float32)
    act = torch.empty((K, L + 1, _lib.UNITS // 4, N * M, 4), device=dev, dtype=torch.float32)
    scratch = torch.empty((N, M), device=dev, dtype=torch.float32)
    _lib.check(
        PROFILE.run("pf_heads_forward_train", 1, lib.mmf_pf_heads_forward_train, C.byref(model_struct), N, M,
                    _lib.ptr(states), _lib.ptr(eps), _lib.ptr(moved), _lib.ptr(rowbias), enabled_mask, precision,
                    _lib.ptr(ll), _lib.ptr(act), _lib.ptr(scratch), _lib.stream_of(states))
    )
    return moved, ll, act


def pf_heads_backward(model_struct, N, M, act, d_ll, enabled_mask):
    """d_ll (K,N,M) -> delta (K,L+1,16,N*M,4) (chunk-major like act): plane l = delta of 64x64 layer l, plane L = delta
    of the input layer."""
    lib = _lib.load()
    act, d_ll = _f32c(act), _f32c(d_ll)
    delta = torch.empty_like(act)  # every plane of every enabled head is fully written by the kernel
    _lib.check(
        PROFILE.run("pf_heads_backward", 1, lib.mmf_pf_heads_backward, C.byref(model_struct), N, M, _lib.ptr(act),
                    _lib.ptr(d_ll), enabled_mask, _lib.ptr(delta), _lib.stream_of(act))
    )
    return delta


def rows_view(t):
    """(..., 16, P, 4) chunk-major planes -> (..., P, 64) row matrices (a copy; for tests and debugging)."""
    return t.transpose(-3, -2).reshape(*t.shape[:-3], t.shape[-2], t.shape[-3] * t.shape[-1])


def pf_heads_weight_grads(act, delta, states, d_ll):
    """act, delta (K, L+1, 16, P, 4), states (P, sd), d_ll (K, P) -> parameter gradients of every head:
    dW (K, L, 64, 64) = delta_l^T a_l, db (K, L+1, 64) = column sums of delta (plane L: the input layer),
    g_in (K, 64, sd) = delta_L^T states, g_out (K, 64) = a_L^T d_ll.  Deterministic: per-CTA partial sums go through a
    workspace and are added in a fixed order (three launches: dW, the two thin end layers, the reduction)."""
    lib = _lib.load()
    K, Lp1, _, P, _ = act.shape
    sd = states.shape[1]
    dev, U = act.device, _lib.UNITS
    dW = torch.empty((K, Lp1 - 1, U, U), device=dev, dtype=torch.float32)
    db = torch.empty((K, Lp1, U), device=dev, dtype=torch.float32)
    g_in = torch.empty((K, U, sd), device=dev, dtype=torch.float32)
    g_out = torch.empty((K, U), device=dev, dtype=torch.float32)
    states, d_ll = _f32c(states), _f32c(d_ll)
    with torch.cuda.device(dev):
        need = lib.mmf_pf_heads_weight_grads_workspace_bytes(K, Lp1 - 1, P)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=dev)  # stream-ordered, graph-capture safe
    _lib.check(
        PROFILE.run("pf_heads_weight_grads", 3, lib.mmf_pf_heads_weight_grads, K, Lp1 - 1, P, sd, _lib.ptr(act),
                    _lib.ptr(delta), _lib.ptr(states), _lib.ptr(d_ll), _lib.ptr(dW), _lib.ptr(db), _lib.ptr(g_in),
                    _lib.ptr(g_out), _lib.ptr(ws), _lib.stream_of(act))
    )
    return dW, db, g_in, g_out


# ---- image encoder trunk ------------------------------------------------------------------------------------
def enc_map_bytes(channels: int) -> int:
    return int(_lib.load().mmf_enc_map_bytes(channels))


def enc_new_map(n_images: int, channels: int, device) -> torch.Tensor:
    """Zero-initialised activation map (bf16 hi/lo planes); the zero guards are never written by the kernels."""
    return torch.zeros(n_images * enc_map_bytes(channels), dtype=torch.uint8, device=device)


def enc_pack_stem(conv) -> torch.Tensor:
    """Conv2d(1, 32, 5) -> fp32 [tap 25][32] + bias[32]."""
    w = conv.weight.detach().float().reshape(32, 25).t().contiguous().reshape(-1)
    return torch.cat([w, conv.bias.detach().float()]).contiguous()


def enc_pack_conv3x3(conv) -> torch.Tensor:
    """Conv2d(cin, cout, 3) -> bf16 [tap][cin/8][2 npad: hi rows then lo rows][8] + fp32 bias[npad] as one byte tensor."""
    w = conv.weight.detach().float()
    cout, cin = w.shape[0], w.shape[1]
    npad = 32 if cout > 16 else 16
    wp = torch.zeros(npad, cin, 3, 3, device=w.device)
    wp[:cout] = w
    hi = wp.to(torch.bfloat16)
    lo = (wp - hi.float()).to(torch.bfloat16)

    def layout(t):  # (npad, cin, 3, 3) -> (tap, cin/8, npad, 8)
        return t.permute(2, 3, 1, 0).reshape(9, cin // 8, 8, npad).permute(0, 1, 3, 2).contiguous()

    # rows [0, npad) = hi, [npad, 2 npad) = lo: one MMA over the stacked rows yields a*w_hi and a*w_lo together
    img = torch.cat([layout(hi), layout(lo)], dim=2).contiguous().view(torch.uint8).reshape(-1)
    bias = torch.zeros(npad, device=w.device)
    bias[:cout] = conv.bias.detach().float()
    return torch.cat([img, bias.view(torch.uint8).reshape(-1)]).contiguous()


def enc_stem(images, w_stem, out_map):
    lib = _lib.load()
    n = images.shape[0]
    _lib.check(PROFILE.run("enc_stem", 1, lib.mmf_enc_stem, n, _lib.ptr(images), _lib.ptr(w_stem), _lib.ptr(out_map),
                           _lib.stream_of(images)))


def enc_conv3x3(n_images, cin, cout, in_map, w_image, *, res_map=None, relu=True, out_map=None, out_nchw=None):
    lib = _lib.load()
    _lib.check(PROFILE.run("enc_conv3x3", 1, lib.mmf_enc_conv3x3, n_images, cin, cout, _lib.ptr(in_map),
                           _lib.ptr(w_image), _lib.ptr(res_map), int(relu), _lib.ptr(out_map), _lib.ptr(out_nchw),
                           _lib.stream_of(in_map)))


def enc_pack_conv3x3_dx(conv) -> torch.Tensor:
    """Conv2d(cin, cout, 3) -> bf16 [dy 3][cin/8][6 npad rows: hi dx-1 | hi dx0 | hi dx+1 | lo dx-1 | lo dx0 | lo dx+1][8]
    + fp32 bias[npad]: the operand image of the dx-stacked trunk kernel (MMF_ENC_VARIANT=3)."""
    w = conv.weight.detach().float()
    cout, cin = w.shape[0], w.shape[1]
    npad = 32 if cout > 16 else 16
    wp = torch.zeros(npad, cin, 3, 3, device=w.device)
    wp[:cout] = w
    hi = wp.to(torch.bfloat16)
    lo = (wp - hi.float()).to(torch.bfloat16)
    t = torch.stack([hi, lo])                                   # (hl, n, c, ky, kx)
    t = t.reshape(2, npad, cin // 8, 8, 3, 3).permute(4, 2, 0, 5, 1, 3)  # (ky, kc, hl, kx, n, j)
    img = t.contiguous().view(torch.uint8).reshape(-1)
    bias = torch.zeros(npad, device=w.device)
    bias[:cout] = conv.bias.detach().float()
    return torch.cat([img, bias.view(torch.uint8).reshape(-1)]).contiguous()


def enc_trunk_variant() -> int:
    return int(os.environ.get("MMF_ENC_VARIANT", "0"))


def enc_pack_trunk(convs) -> torch.Tensor:
    """[stem, block1, block2, 32->16, 16->cout] Conv2d modules -> the weight buffer of mmf_enc_trunk (the layout of
    the 3x3 layers depends on the kernel variant: dx-stacked for variant 3)."""
    stem, c2a, c2b, c3, c4 = convs
    pack = enc_pack_conv3x3_dx if enc_trunk_variant() == 3 else enc_pack_conv3x3
    buf = torch.cat([pack(c2a), pack(c2b), pack(c3), pack(c4),
                     enc_pack_stem(stem).view(torch.uint8).reshape(-1)]).contiguous()
    assert buf.numel() == int(_lib.load().mmf_enc_trunk_weight_bytes())
    return buf


def enc_trunk_scratch(device) -> torch.Tensor:
    return torch.zeros(int(_lib.load().mmf_enc_trunk_scratch_bytes()), dtype=torch.uint8, device=device)


def enc_trunk(images, weights, scratch, cout):
    """images (n, 32, 32) fp32 -> (n, cout, 32, 32) fp32: the whole convolutional trunk in one launch."""
    lib = _lib.load()
    n = images.shape[0]
    out = torch.empty((n, cout, 32, 32), device=images.device, dtype=torch.float32)
    _lib.check(PROFILE.run("enc_trunk", 1, lib.mmf_enc_trunk, n, cout, _lib.ptr(images), _lib.ptr(weights),
                           _lib.ptr(scratch), _lib.ptr(out), _lib.stream_of(images)))
    return out


def row_mlp(program_ops, weights, inputs, in_slots, out_dims, out_slots, scratch):
    """One launch of a compiled per-trajectory MLP program (``fused.RowProgram``): inputs are (rows, d_i) fp32 tensors,
    returns the list of (rows, out_dims[i]) outputs."""
    lib = _lib.load()
    rows = inputs[0].shape[0]
    inputs = [_f32c(x) for x in inputs]
    assert all(x.dim() == 2 and x.shape[0] == rows for x in inputs)
    dev = inputs[0].device
    outs = [torch.empty((rows, d), device=dev, dtype=torch.float32) for d in out_dims]
    n_ops, n_in, n_out = len(program_ops), len(inputs), len(outs)
    op_arr = (_lib.MlpOp * n_ops)(*program_ops)
    in_ptrs = (C.c_void_p * n_in)(*[x.data_ptr() for x in inputs])
    in_dims = (C.c_int32 * n_in)(*[x.shape[1] for x in inputs])
    in_sl = (C.c_int32 * n_in)(*in_slots)
    out_ptrs = (C.c_void_p * n_out)(*[o.data_ptr() for o in outs])
    out_d = (C.c_int32 * n_out)(*out_dims)
    out_sl = (C.c_int32 * n_out)(*out_slots)
    for x in inputs:  # devices of the buffers whose pointers travel in arrays
        _lib.ptr(x)
    _lib.check(PROFILE.run("row_mlp", 1, lib.mmf_row_mlp, rows, op_arr, n_ops, _lib.ptr(weights), in_ptrs, in_dims, in_sl,
                           n_in, out_ptrs, out_d, out_sl, n_out, scratch, _lib.stream_of(inputs[0])))
    return outs


def pf_init(mean, covariance, eps_MNsd):
    """R2: (N,sd), (N,sd,sd), (M,N,sd) -> particle_states (N,M,sd), particle_log_weights (N,M)."""
    lib = _lib.load()
    M, N, sd = eps_MNsd.shape
    assert mean.shape == (N, sd) and covariance.shape == (N, sd, sd)
    mean, covariance, eps_MNsd = _f32c(mean), _f32c(covariance), _f32c(eps_MNsd)
    states = torch.empty((N, M, sd), device=mean.device, dtype=torch.float32)
    logw = torch.empty((N, M), device=mean.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("pf_init", 1, lib.mmf_pf_init, N, M, sd, _lib.ptr(mean), _lib.ptr(covariance), _lib.ptr(eps_MNsd), _lib.ptr(states),
                        _lib.ptr(logw), _lib.stream_of(mean))
    )
    return states, logw


def pf_traj_rows(model_struct, K, controls, obs_feats):
    """Hoisted per-trajectory rows: controls (N,cd), obs_feats list of K tensors (N,F_k) or None."""
    lib = _lib.load()
    controls = _f32c(controls)
    N = controls.shape[0]
    feats = [None if f is None else _f32c(f) for f in obs_feats]
    arr = (C.c_void_p * _lib.MAX_HEADS)()
    for k in range(K):
        arr[k] = None if feats[k] is None else feats[k].data_ptr()
    out = torch.empty((1 + K, N, _lib.UNITS), device=controls.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("pf_traj_rows", 1, lib.mmf_pf_traj_rows, C.byref(model_struct), N, _lib.ptr(controls), arr, _lib.ptr(out), _lib.stream_of(controls))
    )
    return out


def pf_predict_measure(model_struct, states, eps, rowbias, logw, modality_logw, enabled_mask, precision=PREC_FP32,
                       want_ll=False):
    """R3+R4+R5: states (N,M,sd), eps (N*M,sd), rowbias (1+K,N,64), logw (N,M), modality_logw (N,K)|None
    -> states_new (N,M,sd), logw_unnorm (N,M) [, ll (K,N,M)]."""
    lib = _lib.load()
    N, M, sd = states.shape
    states, eps, rowbias, logw = _f32c(states), _f32c(eps), _f32c(rowbias), _f32c(logw)
    assert eps.numel() == N * M * sd and logw.shape == (N, M)
    K = model_struct.num_heads
    assert rowbias.shape == (1 + K, N, _lib.UNITS), f"rowbias {tuple(rowbias.shape)} != {(1 + K, N, _lib.UNITS)}"
    if modality_logw is not None:
        modality_logw = _f32c(modality_logw)
        assert modality_logw.shape == (N, K), (modality_logw.shape, (N, K))
    states_out = torch.empty_like(states)
    logw_out = torch.empty_like(logw)
    ll = torch.full((K, N, M), float("nan"), device=states.device, dtype=torch.float32) if want_ll else None
    _lib.check(
        PROFILE.run(
            "pf_predict_measure", 1, lib.mmf_pf_predict_measure,
            C.byref(model_struct), N, M, _lib.ptr(states), _lib.ptr(eps), _lib.ptr(rowbias), _lib.ptr(logw),
            _lib.ptr(modality_logw), enabled_mask, precision, _lib.ptr(states_out), _lib.ptr(logw_out),
            _lib.ptr(ll), _lib.stream_of(states),
        )
    )
    return (states_out, logw_out, ll) if want_ll else (states_out, logw_out)


def pf_forward_loop(model_struct, states, logw, controls, feats, modality_logw, enabled_mask, eps, *, precision,
                    estimation, mode, uniforms):
    """R1: the whole T-step recursion in one C call (1 + 2 T kernel launches; small problems -- M <= 128, N up to two CTAs
    per SM -- 2 launches: the per-trajectory rows and the one-launch whole-sequence kernel, fp32 arithmetic).  states (N,M,sd) and logw (N,M) are
    UPDATED IN PLACE to the particle set after the last step; controls (T,N,cd), feats: K tensors (T,N,F_k) or None,
    modality_logw (T,N,K)|None, eps (T,N*M,sd), uniforms float64 (T,N,M) | (T,N) | None.  Returns estimates (T,N,sd)."""
    lib = _lib.load()
    N, M, sd = states.shape
    T = controls.shape[0]
    K = model_struct.num_heads
    assert states.dtype == torch.float32 and states.is_contiguous() and logw.is_contiguous() and logw.shape == (N, M)
    controls, eps = _f32c(controls), _f32c(eps)
    assert controls.shape[:2] == (T, N) and eps.numel() == T * N * M * sd
    feats = [None if f is None else _f32c(f) for f in feats]
    assert len(feats) == K and all(f is None or f.shape[:2] == (T, N) for f in feats), "observation features / (T, N) mismatch"
    arr = (C.c_void_p * _lib.MAX_HEADS)()
    for k in range(K):
        arr[k] = None if feats[k] is None else feats[k].data_ptr()
    if modality_logw is not None:
        modality_logw = _f32c(modality_logw)
        assert modality_logw.shape == (T, N, K), (modality_logw.shape, (T, N, K))
    dev = states.device
    if mode != RESAMPLE_NONE:
        assert uniforms is not None and uniforms.dtype == torch.float64
        uniforms = uniforms.contiguous()
        assert uniforms.shape == ((T, N) if is_systematic(mode) else (T, N, M)), uniforms.shape
    rowbias = torch.empty((1 + K, T * N, _lib.UNITS), device=dev, dtype=torch.float32)
    states_ws, logw_ws = torch.empty_like(states), torch.empty_like(logw)
    est = torch.empty((T, N, sd), device=dev, dtype=torch.float32)
    ws = _resample_workspace(N, M, dev)
    for f in feats:  # note the feature tensors' device for the launch guard (their pointers travel in `arr`)
        _lib.ptr(f)
    _lib.check(
        PROFILE.run(
            "pf_forward_loop", 2 if lib.mmf_pf_forward_loop_persistent(N, M) else 1 + 2 * T, lib.mmf_pf_forward_loop, C.byref(model_struct), T, N, M, _lib.ptr(states),
            _lib.ptr(logw), _lib.ptr(controls), arr, _lib.ptr(modality_logw), enabled_mask, precision, _lib.ptr(eps),
            estimation, mode, _lib.ptr(uniforms), _lib.ptr(rowbias), _lib.ptr(states_ws), _lib.ptr(logw_ws), _lib.ptr(est),
            _lib.ptr(ws), _lib.stream_of(states),
        )
    )
    return est


def _resample_workspace(N, M, device):
    """Global scratch for trajectories that do not fit shared memory.  Allocated per call from torch's stream-ordered
    caching allocator: two streams never share a slice, and during CUDA-graph capture the buffer comes from (and stays
    alive in) the graph's private pool, so a replayed graph never writes into memory that has been handed to someone
    else."""
    with torch.cuda.device(device):
        need = _lib.load().mmf_pf_resample_workspace_bytes(N, M)
    if need == 0:
        return None
    return torch.empty(need, dtype=torch.uint8, device=device)


def pf_normalize_resample(states, logw_unnorm, *, estimation=ESTIMATE_WEIGHTED_AVERAGE, mode=RESAMPLE_NONE,
                          alpha=1.0, M_out=None, uniforms=None, want_debug=False):
    """Second half of R6 + R7.  Returns dict(states, logw, estimate[, logw_norm, logits, idx])."""
    lib = _lib.load()
    N, M, sd = states.shape
    states, logw_unnorm = _f32c(states), _f32c(logw_unnorm)
    assert logw_unnorm.shape == (N, M)
    dev = states.device
    est = torch.empty((N, sd), device=dev, dtype=torch.float32)
    resample = mode != RESAMPLE_NONE
    if resample:
        M_out = M if M_out is None else M_out
        assert uniforms is not None and uniforms.dtype == torch.float64
        uniforms = uniforms.contiguous()
        assert uniforms.shape == ((N,) if is_systematic(mode) else (N, M_out)), uniforms.shape
        states_out = torch.empty((N, M_out, sd), device=dev, dtype=torch.float32)
        logw_out = torch.empty((N, M_out), device=dev, dtype=torch.float32)
    else:
        M_out = M
        states_out = None
        logw_out = torch.empty((N, M), device=dev, dtype=torch.float32)
    logw_norm = torch.empty((N, M), device=dev, dtype=torch.float32) if want_debug else None
    logits = torch.empty((N, M), device=dev, dtype=torch.float32) if (want_debug and resample) else None
    idx = torch.empty((N, M_out), device=dev, dtype=torch.int64) if (want_debug and resample) else None
    ws = _resample_workspace(N, M, dev)
    _lib.check(
        PROFILE.run(
            "pf_normalize_resample", 1, lib.mmf_pf_normalize_resample,
            N, M, sd, _lib.ptr(states), _lib.ptr(logw_unnorm), estimation, mode, float(alpha), M_out,
            _lib.ptr(uniforms), _lib.ptr(states_out), _lib.ptr(logw_out), _lib.ptr(est), _lib.ptr(logw_norm),
            _lib.ptr(logits), _lib.ptr(idx), _lib.ptr(ws), _lib.stream_of(states),
        )
    )
    out = {"states": states_out if resample else states, "logw": logw_out, "estimate": est}
    if want_debug:
        out.update(logw_norm=logw_norm, logits=logits, idx=idx)
    return out


def fuse_loglik(ll, w=None):
    """R5 standalone: ll (N,M,K), w (N,K)|None -> (N,M)."""
    lib = _lib.load()
    N, M, K = ll.shape
    ll = _f32c(ll)
    w = None if w is None else _f32c(w)
    out = torch.empty((N, M), device=ll.device, dtype=torch.float32)
    _lib.check(PROFILE.run("fuse_loglik", 1, lib.mmf_fuse_loglik, N, M, K, _lib.ptr(ll), _lib.ptr(w), _lib.ptr(out), _lib.stream_of(ll)))
    return out


def resample_indices(logits, uniforms, mode=RESAMPLE_MULTINOMIAL_STRICT, M_out=None):
    """R7 standalone: logits (N,M), float64 uniforms -> int64 (N,M_out)."""
    lib = _lib.load()
    N, M = logits.shape
    logits = _f32c(logits)
    assert uniforms.dtype == torch.float64
    uniforms = uniforms.contiguous()
    if M_out is None:
        M_out = M if is_systematic(mode) else uniforms.shape[1]
    idx = torch.empty((N, M_out), device=logits.device, dtype=torch.int64)
    ws = _resample_workspace(N, M, logits.device)
    _lib.check(
        PROFILE.run("resample", 1, lib.mmf_resample, N, M, M_out, _lib.ptr(logits), mode, _lib.ptr(uniforms), _lib.ptr(idx), _lib.ptr(ws),
                         _lib.stream_of(logits))
    )
    return idx


def ekf_loop(model_structs, mean0, cov0, controls, z, r_tril):
    """R8 for F filters x T steps: mean0 (F,N,sd), cov0 (F,N,sd,sd), controls (T,N,cd), z (F,T,N,sd),
    r_tril (F,T,N,sd,sd) -> means (F,T,N,sd), covs (F,T,N,sd,sd)."""
    lib = _lib.load()
    F = len(model_structs)
    arr = (_lib.EKFModel * F)(*model_structs)
    mean0, cov0, controls, z, r_tril = map(_f32c, (mean0, cov0, controls, z, r_tril))
    _, T, N, sd = z.shape
    assert mean0.shape == (F, N, sd) and cov0.shape == (F, N, sd, sd)
    assert controls.shape[:2] == (T, N) and r_tril.shape == (F, T, N, sd, sd)
    means = torch.empty((F, T, N, sd), device=z.device, dtype=torch.float32)
    covs = torch.empty((F, T, N, sd, sd), device=z.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("ekf_loop", 1, lib.mmf_ekf_loop_fwd, arr, F, T, N, _lib.ptr(mean0), _lib.ptr(cov0), _lib.ptr(controls), _lib.ptr(z),
                             _lib.ptr(r_tril), _lib.ptr(means), _lib.ptr(covs), _lib.stream_of(z))
    )
    return means, covs


def ekf_loop_train(model_structs, mean0, cov0, controls, z, r_tril):
    """``ekf_loop`` that also records the tape of ``ekf_loop_bwd``: -> means (F,T,N,sd), covs (F,T,N,sd,sd),
    pred (F,T,N,sd) = mu- and jac (F,T,N,sd,sd) = A of every step.  means / covs equal ``ekf_loop``'s bit for bit."""
    lib = _lib.load()
    F = len(model_structs)
    arr = (_lib.EKFModel * F)(*model_structs)
    mean0, cov0, controls, z, r_tril = map(_f32c, (mean0, cov0, controls, z, r_tril))
    _, T, N, sd = z.shape
    assert mean0.shape == (F, N, sd) and cov0.shape == (F, N, sd, sd)
    assert controls.shape[:2] == (T, N) and r_tril.shape == (F, T, N, sd, sd)
    means = torch.empty((F, T, N, sd), device=z.device, dtype=torch.float32)
    covs = torch.empty((F, T, N, sd, sd), device=z.device, dtype=torch.float32)
    pred = torch.empty_like(means)
    jac = torch.empty_like(covs)
    _lib.check(
        PROFILE.run("ekf_loop_train", 1, lib.mmf_ekf_loop_train_fwd, arr, F, T, N, _lib.ptr(mean0), _lib.ptr(cov0),
                    _lib.ptr(controls), _lib.ptr(z), _lib.ptr(r_tril), _lib.ptr(means), _lib.ptr(covs), _lib.ptr(pred),
                    _lib.ptr(jac), _lib.stream_of(z))
    )
    return means, covs, pred, jac


def ekf_loop_bwd(model_structs, cov0, z, r_tril, covs, pred, jac, d_means=None, d_covs=None):
    """Reverse mode of ``ekf_loop_train`` (frozen dynamics, A a constant of the recursion): the forward's inputs and
    outputs plus d_means (F,T,N,sd) | None, d_covs (F,T,N,sd,sd) | None -> d_mean0, d_cov0, d_z, d_r_tril."""
    lib = _lib.load()
    F = len(model_structs)
    arr = (_lib.EKFModel * F)(*model_structs)
    cov0, z, r_tril, covs, pred, jac = map(_f32c, (cov0, z, r_tril, covs, pred, jac))
    _, T, N, sd = z.shape
    assert cov0.shape == (F, N, sd, sd) and r_tril.shape == covs.shape == jac.shape == (F, T, N, sd, sd)
    assert pred.shape == z.shape
    d_means = None if d_means is None else _f32c(d_means)
    d_covs = None if d_covs is None else _f32c(d_covs)
    assert d_means is None or d_means.shape == z.shape
    assert d_covs is None or d_covs.shape == covs.shape
    dev = z.device
    d_mean0 = torch.empty((F, N, sd), device=dev, dtype=torch.float32)
    d_cov0 = torch.empty_like(cov0)
    d_z = torch.empty_like(z)
    d_r = torch.empty_like(r_tril)
    _lib.check(
        PROFILE.run("ekf_loop_bwd", 1, lib.mmf_ekf_loop_bwd, arr, F, T, N, None, _lib.ptr(cov0), _lib.ptr(z),
                    _lib.ptr(r_tril), None, _lib.ptr(covs), _lib.ptr(pred), _lib.ptr(jac), _lib.ptr(d_means),
                    _lib.ptr(d_covs), _lib.ptr(d_mean0), _lib.ptr(d_cov0), _lib.ptr(d_z), _lib.ptr(d_r),
                    _lib.stream_of(z))
    )
    return d_mean0, d_cov0, d_z, d_r


def dynamics_jacobian(model_struct, states, controls):
    """A.4: states (N,sd), controls (N,cd) -> pred (N,sd), jacobian (N,sd,sd)."""
    lib = _lib.load()
    states, controls = _f32c(states), _f32c(controls)
    N, sd = states.shape
    pred = torch.empty_like(states)
    jac = torch.empty((N, sd, sd), device=states.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("dynamics_jacobian", 1, lib.mmf_dynamics_jacobian, C.byref(model_struct), N, _lib.ptr(states), _lib.ptr(controls), _lib.ptr(pred),
                                  _lib.ptr(jac), _lib.stream_of(states))
    )
    return pred, jac


def kf_fuse_crossmodal(mu, P, beta):
    """R10: mu (K,*,sd), P (K,*,sd,sd), beta (K,*,sd) -> mean (*,sd), cov (*,sd,sd)."""
    lib = _lib.load()
    K, sd = mu.shape[0], mu.shape[-1]
    lead = mu.shape[1:-1]
    rows = int(math.prod(lead))
    mu, P, beta = _f32c(mu), _f32c(P), _f32c(beta)
    mean = torch.empty((*lead, sd), device=mu.device, dtype=torch.float32)
    cov = torch.empty((*lead, sd, sd), device=mu.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("kf_fuse_crossmodal", 1, lib.mmf_kf_fuse_crossmodal, K, rows, sd, _lib.ptr(mu), _lib.ptr(P), _lib.ptr(beta), _lib.ptr(mean),
                                   _lib.ptr(cov), _lib.stream_of(mu))
    )
    return mean, cov


def pf_reweight_train_fwd(ll, modality_logw, logw_in, states, enabled_mask):
    """R5 + R6 of the BPTT step: ll (K,N,M), modality_logw (N,K)|None, logw_in (N,M), states (N,M,sd) ->
    normalised log-weights (N,M), weighted-average estimate (N,sd)."""
    lib = _lib.load()
    K, N, M = ll.shape
    sd = states.shape[-1]
    ll, logw_in, states = _f32c(ll), _f32c(logw_in), _f32c(states)
    modality_logw = None if modality_logw is None else _f32c(modality_logw)
    assert logw_in.shape == (N, M) and states.shape == (N, M, sd) and (modality_logw is None or modality_logw.shape == (N, K))
    logw = torch.empty((N, M), device=ll.device, dtype=torch.float32)
    est = torch.empty((N, sd), device=ll.device, dtype=torch.float32)
    _lib.check(PROFILE.run("pf_reweight_train_fwd", 1, lib.mmf_pf_reweight_train_fwd, N, M, K, sd, enabled_mask, _lib.ptr(ll),
                           _lib.ptr(modality_logw), _lib.ptr(logw_in), _lib.ptr(states), _lib.ptr(logw), _lib.ptr(est),
                           _lib.stream_of(ll)))
    return logw, est


def pf_reweight_train_bwd(ll, modality_logw, logw_in, states, enabled_mask, d_est, d_logw):
    """Reverse mode of ``pf_reweight_train_fwd``: -> d_ll (K,N,M), d_modality_logw (N,K)|None, d_logw_in (N,M)."""
    lib = _lib.load()
    K, N, M = ll.shape
    sd = states.shape[-1]
    d_est = None if d_est is None else _f32c(d_est)
    d_logw = None if d_logw is None else _f32c(d_logw)
    d_ll = torch.empty((K, N, M), device=ll.device, dtype=torch.float32)
    d_w = None if modality_logw is None else torch.empty((N, K), device=ll.device, dtype=torch.float32)
    d_in = torch.empty((N, M), device=ll.device, dtype=torch.float32)
    _lib.check(PROFILE.run("pf_reweight_train_bwd", 1, lib.mmf_pf_reweight_train_bwd, N, M, K, sd, enabled_mask, _lib.ptr(ll),
                           _lib.ptr(modality_logw), _lib.ptr(logw_in), _lib.ptr(states), _lib.ptr(d_est), _lib.ptr(d_logw),
                           _lib.ptr(d_ll), _lib.ptr(d_w), _lib.ptr(d_in), _lib.stream_of(ll)))
    return d_ll, d_w, d_in


def kf_fuse_measurements(z, r_tril, weights=None):
    """R12: z (K,*,sd), r_tril (K,*,sd,sd), weights (K,*,sd) or None (unimodal) -> fused z (*,sd) and a lower factor
    (crossmodal) / covariance (unimodal) (*,sd,sd)."""
    lib = _lib.load()
    K, sd = z.shape[0], z.shape[-1]
    lead = z.shape[1:-1]
    rows = int(math.prod(lead))
    z, r_tril = _f32c(z), _f32c(r_tril)
    if weights is not None:
        weights = _f32c(weights)
        assert weights.shape == z.shape
    assert r_tril.shape == (K, *lead, sd, sd)
    z_out = torch.empty((*lead, sd), device=z.device, dtype=torch.float32)
    mat = torch.empty((*lead, sd, sd), device=z.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("kf_fuse_measurements", 1, lib.mmf_kf_fuse_measurements, K, rows, sd, _lib.ptr(z), _lib.ptr(r_tril),
                    None if weights is None else _lib.ptr(weights), _lib.ptr(z_out), _lib.ptr(mat), _lib.stream_of(z))
    )
    return z_out, mat


def kf_fuse_unimodal(mu, P):
    """R11: information-form fusion of K Gaussian posteriors."""
    lib = _lib.load()
    K, sd = mu.shape[0], mu.shape[-1]
    lead = mu.shape[1:-1]
    rows = int(math.prod(lead))
    mu, P = _f32c(mu), _f32c(P)
    mean = torch.empty((*lead, sd), device=mu.device, dtype=torch.float32)
    cov = torch.empty((*lead, sd, sd), device=mu.device, dtype=torch.float32)
    _lib.check(
        PROFILE.run("kf_fuse_unimodal", 1, lib.mmf_kf_fuse_unimodal, K, rows, sd, _lib.ptr(mu), _lib.ptr(P), _lib.ptr(mean), _lib.ptr(cov),
                                 _lib.stream_of(mu))
    )
    return mean, cov
