"""The fused BPTT kernels at the size the project trains at (BASELINE config C4: PushCrossmodalParticleFilter, N = 8192
trajectories x M = 30 particles, P = N M = 245,760 particle rows per step), against float64.

At the 1,920 rows of the other training tests none of the kernels runs the code C4 needs:

    k_particle_chain_ws<4,2,true>  forward + saved activations; a group loops over a second tile only when
                                   P > 4 groups x SMs x 128 rows, overlapping the next tile's input layer with the
                                   output-layer MMA of the current one; the issuer's last slot may hold < 4 tiles
    k_head_chain_bwd<4>            deltas; the same tile loop, its mbarrier phase carried from tile to tile
    k_heads_dw_tc                  dW = delta^T act over 64-row tiles of a row chunk, double-buffered operands: the
                                   buffers are reused (wait, parity flip, drain) only from a CTA's third tile on
    k_heads_edge_grads, k_heads_grads_reduce   the thin end layers and the fixed-order reduction

Every shape below restates the launchers' grid arithmetic (and the weight-gradient row partition) in Python and asserts
the regime it is meant for before it runs, and torch.profiler confirms the kernel that ran.  References:

  * forward: moved states through the float64 dynamics chain end to end; every activation plane teacher-forced layer by
    layer from the kernel's own previous plane (so one layer's error cannot compound); ll from the kernel's own last plane;
  * backward: float64 autograd through the chain with every ReLU replaced by its mask (kernel activation > 0): linear in
    d_ll, so no ReLU can flip and what is left is the kernel's split-bf16 arithmetic;
  * weight gradients: small-integer inputs, for which the split bf16 operands are exact (lo = 0) and every fp32 partial
    sum is an integer below 2^24, so the kernel must equal the float64 reference bit for bit;
  * the whole training step at C4 size against the oracle port evaluated in float64 on the GPU.

Outputs are prefilled with NaN (the workspace too): a row or plane a kernel never writes fails the comparison.
"""
import ctypes as C
import math
import time

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import crossmodal_port as port  # noqa: E402
from oracle.noise import RecordedNoise  # noqa: E402

from multimodalfilter_b200 import _lib, fused, ops  # noqa: E402
from multimodalfilter_b200.crossmodal import models as M  # noqa: E402
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories  # noqa: E402

from full_size import (  # noqa: E402
    GROUPS, TILE, assert_rows, chain_layers, chain_regime, dynamics_moved, nm_for_tiles, profiled)
from util import ReplayNoise, draw_noise  # noqa: E402

DEV = "cuda:0"
U = _lib.UNITS
DWT_ROWS = 64                # k_heads_dw_tc: rows per tile
C4_N, C4_M = 8192, 30
FWD = "k_particle_chain_ws<4,2,true>"
BWD = "k_head_chain_bwd<4>"
DW = ("k_heads_dw_tc", "k_heads_edge_grads", "k_heads_grads_reduce")
# Bars.  Moved states and ll: 1e-4 for bf16x3, the parity bar of the forward (test_predict_measure_matches_oracle_modules),
# and 3e-2 for single-pass bf16, the grade that test holds it to.  The activation planes and the deltas are compared entry
# by entry over 15.7 M entries per plane here, against 22 k in test_heads_backward_kernel_matches_autograd; the split-bf16
# rounding error is spread like a Gaussian, whose expected maximum grows as sqrt(2 ln n): 1.3x from there to here.
# Measured on a B200 (1000 W power limit), worst over every case below: planes 1.16e-4 (bf16x3) and 3.3e-2 (bf16), deltas
# 2.8e-4 (delta 0, seven layers of backward from d_ll).  The bars are those of the small tests times 2 (planes) and 2.5
# (deltas); a misplaced row or tile is wrong by O(1).
RTOL_X3 = 1e-4
RTOL_BF16 = 3e-2
RTOL_PLANE_X3 = 2e-4
RTOL_PLANE_BF16 = 6e-2
RTOL_DELTA = 5e-4
MODELS = {"push": ("PushCrossmodalParticleFilter", 2), "door": ("DoorCrossmodalParticleFilter", 3)}


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the launchers' arithmetic, restated ----------------------------------------------------------------------------
def dw_partition(K, L, P, sms):
    """particle_chain_bwd.cu dw_partition: (dw_chunks, dw_rows, edge_chunks, edge_rows)."""
    chunks = (sms * 3 + K * L - 1) // (K * L)
    rows = -(-P // chunks)
    rows = -(-rows // DWT_ROWS) * DWT_ROWS
    chunks = -(-P // rows)
    e_chunks = (sms * 4 + K - 1) // K
    e_rows = -(-P // e_chunks)
    e_rows = -(-e_rows // 16) * 16
    e_chunks = -(-P // e_rows)
    return chunks, rows, e_chunks, e_rows


def dw_regime(K, L, P, sms):
    chunks, rows, _, _ = dw_partition(K, L, P, sms)
    last = P - rows * (chunks - 1)
    return {"chunks": chunks, "tiles_per_chunk": rows // DWT_ROWS, "last_chunk_rows": last,
            "last_chunk_tiles": -(-last // DWT_ROWS), "ragged": last % DWT_ROWS != 0}


def chain_shapes(sms):
    """C4 itself, and tiles = 4 SMs k + r (r = 1, 2, 3): k full sweeps of the grid, then a last slot of r tiles whose last
    tile is ragged."""
    out = {"c4": (C4_N, C4_M)}
    for r, k in ((1, 1), (2, 2), (3, 1)):
        out[f"sweeps{k}+{r}"] = nm_for_tiles(GROUPS * sms * k + r, 37)
    return out


def assert_chain_regime(case, P, sms):
    g = chain_regime(P, sms)
    if case == "c4":
        assert P == 245760 and g["ctas"] == sms and g["tiles_per_group"] >= 2, g
        assert g["tiles"] > GROUPS * sms  # some groups loop over a second tile
    else:
        k, r = (int(v) for v in case[len("sweeps"):].split("+"))
        assert g["tiles"] == GROUPS * sms * k + r and g["ctas"] == sms, g
        assert g["tiles_per_group"] == k + 1 and g["last_slot"] == r and 0 < g["last_tile_rows"] < TILE, g
    return g


# ---- raw entry points with NaN-prefilled outputs -------------------------------------------------------------------
def forward_train(plan, states, eps, rowbias, mask, precision):
    N, Mp, sd = states.shape
    K, L, P = plan.K, ops.head_depth(plan.struct), N * Mp
    nan = float("nan")
    moved = torch.full_like(states, nan)
    ll = torch.full((K, N, Mp), nan, device=DEV)
    act = torch.full((K, L + 1, U // 4, P, 4), nan, device=DEV)
    scratch = torch.full((N, Mp), nan, device=DEV)
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_pf_heads_forward_train, C.byref(plan.struct), N, Mp, _lib.ptr(states), _lib.ptr(eps),
                         _lib.ptr(moved), _lib.ptr(rowbias), mask, ops.PRECISIONS[precision], _lib.ptr(ll), _lib.ptr(act),
                         _lib.ptr(scratch), _lib.stream_of(states)))
    return moved, ll, act


def heads_backward(plan, N, Mp, act, d_ll, mask):
    delta = torch.full_like(act, float("nan"))
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_pf_heads_backward, C.byref(plan.struct), N, Mp, _lib.ptr(act), _lib.ptr(d_ll), mask,
                         _lib.ptr(delta), _lib.stream_of(act)))
    return delta


def weight_grads(act, delta, x, d_ll):
    K, Lp1, _, P, _ = act.shape
    sd = x.shape[1]
    nan = float("nan")
    outs = [torch.full(s, nan, device=DEV) for s in ((K, Lp1 - 1, U, U), (K, Lp1, U), (K, U, sd), (K, U))]
    lib = _lib.load()
    ws = torch.full((max(lib.mmf_pf_heads_weight_grads_workspace_bytes(K, Lp1 - 1, P), 16),), 0xFF, dtype=torch.uint8,
                    device=DEV)  # all-ones bytes: every float of the workspace is a NaN
    _lib.check(_lib.call(lib.mmf_pf_heads_weight_grads, K, Lp1 - 1, P, sd, _lib.ptr(act), _lib.ptr(delta), _lib.ptr(x),
                         _lib.ptr(d_ll), *(_lib.ptr(o) for o in outs), _lib.ptr(ws), _lib.stream_of(act)))
    return outs


def _plan(model, seed=71):
    name, sd = MODELS[model]
    f = fill_parameters(getattr(M, name)(), seed=seed).to(DEV)
    plan = fused.PFPlan.build(f)
    plan.refresh(torch.device(DEV), backward=True)
    return f, plan, sd


# ---- forward-train and backward kernels against float64 -------------------------------------------------------------
def _fwd_cases():
    cases = []
    for model in MODELS:
        for shape in ("c4", "sweeps1+1", "sweeps2+2", "sweeps1+3"):
            for mask in (0b11, 0b01, 0b10):
                cases.append((model, shape, mask, "bf16x3"))
        cases.append((model, "c4", 0b11, "bf16"))
    return cases


@pytest.mark.parametrize("model,shape,mask,precision", _fwd_cases())
def test_chain_kernels_match_float64(model, shape, mask, precision):
    """mmf_pf_heads_forward_train and mmf_pf_heads_backward at C4 and at tiles = 4 SMs k + r: moved states, every
    activation plane, ll and every delta plane (the input layer's too) against float64, worst error reported per row;
    planes of disabled heads must stay NaN (FusedHeads relies on that)."""
    sms = _sms()
    N, Mp = chain_shapes(sms)[shape]
    P = N * Mp
    assert_chain_regime(shape, P, sms)
    _, plan, sd = _plan(model)
    K, L = plan.K, ops.head_depth(plan.struct)
    g = torch.Generator(device=DEV).manual_seed(P + mask)
    states = torch.randn(N, Mp, sd, device=DEV, generator=g)
    eps = torch.randn(P, sd, device=DEV, generator=g)
    rowbias = torch.randn(1 + K, N, U, device=DEV, generator=g)
    d_ll = torch.randn(K, N, Mp, device=DEV, generator=g)
    moved, ll, act = profiled(lambda: forward_train(plan, states, eps, rowbias, mask, precision), [FWD])
    delta = profiled(lambda: heads_backward(plan, N, Mp, act, d_ll, mask), [BWD])
    bar = RTOL_X3 if precision == "bf16x3" else RTOL_BF16
    plane_bar = RTOL_PLANE_X3 if precision == "bf16x3" else RTOL_PLANE_BF16
    report = {}
    assert_rows(moved.reshape(P, sd), dynamics_moved(plan, states, eps, rowbias[0], Mp), bar, "moved states", report,
                "moved")
    x = moved.reshape(P, sd).double()
    for k, spec in enumerate(plan.heads):
        if not (mask >> k) & 1:
            assert torch.isnan(act[k]).all() and torch.isnan(ll[k]).all(), f"head {k} is disabled but was written"
            assert torch.isnan(delta[k]).all(), f"head {k} is disabled but its deltas were written"
            continue
        (Wi, bi), layers, (Wo, bo) = chain_layers(spec.state, spec.shared, slice(spec.feat_dim, spec.feat_dim + U))
        assert len(layers) == L
        A = ops.rows_view(act[k])  # (L + 1, P, 64)
        rb = rowbias[1 + k].double().repeat_interleave(Mp, dim=0)
        # forward, teacher-forced: plane 0 from the kernel's moved states, plane l + 1 from the kernel's planes l (and l - 1)
        assert_rows(A[0], torch.relu(x @ Wi.T + bi), plane_bar, f"head {k} plane 0", report, "planes")
        for l, (W, b, kind) in enumerate(layers):
            a = A[l].double()
            z = a @ W.T + (rb if kind == "MID" else b)
            if kind == "B":
                z = z + A[l - 1].double()
            assert_rows(A[l + 1], torch.relu(z), plane_bar, f"head {k} plane {l + 1}", report, "planes")
        assert_rows(ll[k].reshape(P, 1), A[L].double() @ Wo.T + bo, bar, f"head {k} ll", report, "ll")
        # backward: float64 autograd through the chain with each ReLU replaced by the kernel's mask (act > 0)
        masks = [(A[i] > 0).double() for i in range(L + 1)]
        z0 = (x @ Wi.T + bi).requires_grad_(True)
        zs = [z0]
        h, res = z0 * masks[0], None
        for l, (W, b, kind) in enumerate(layers):
            z = h @ W.T + (rb if kind == "MID" else b)
            if kind == "B":
                z = z + res
            if kind == "A":
                res = h
            z.retain_grad()
            zs.append(z)
            h = z * masks[l + 1]
        ((h @ Wo.T + bo)[:, 0] * d_ll[k].reshape(P).double()).sum().backward()
        D = ops.rows_view(delta[k])
        for l in range(L):
            assert_rows(D[l], zs[1 + l].grad, RTOL_DELTA, f"head {k} delta {l}", report, "deltas")
        assert_rows(D[L], z0.grad, RTOL_DELTA, f"head {k} input-layer delta", report, "deltas")
        del zs, masks, A, D
    print(f"[{model} {shape} mask={mask:#04b} {precision}] P={P}: worst relative errors "
          + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- weight gradients in exact arithmetic ---------------------------------------------------------------------------
def _dw_cases():
    """(K, head model, sd, regime): every regime is searched for in the row partition of the device at test time."""
    return [(1, "push", 1, "1 tile/chunk, ragged"), (2, "door", 2, "1 tile/chunk, last chunk 1 row"),
            (3, "push", 3, "2 tiles/chunk, ragged"), (1, "door", 4, "2 tiles/chunk, last chunk 1 row"),
            (2, "push", 4, "3 tiles/chunk, ragged"), (3, "door", 1, "3 tiles/chunk, last chunk 1 row"),
            (2, "push", 2, "c4"), (1, "push", 3, "4 tiles/chunk, ragged"), (3, "push", 2, "6 tiles/chunk, last chunk 1 row"),
            (2, "door", 3, "P < 64"), (3, "push", 4, "P = 1")]


def _head_depth(model):
    _, plan, _ = _plan(model)
    return ops.head_depth(plan.struct)


def find_rows(K, L, regime, sms):
    if regime == "c4":
        return C4_N * C4_M
    if regime == "P < 64":
        return 37
    if regime == "P = 1":
        return 1
    t = int(regime.split()[0])
    one_row = regime.endswith("1 row")
    chunks0 = (sms * 3 + K * L - 1) // (K * L)
    for P in range(DWT_ROWS * t * (chunks0 - 1), DWT_ROWS * t * (chunks0 + 1)):
        q = dw_regime(K, L, P, sms)
        if q["chunks"] >= 2 and q["tiles_per_chunk"] == t and (q["last_chunk_rows"] == 1 if one_row else
                                                                 q["ragged"] and q["last_chunk_tiles"] == t):
            return P
    raise AssertionError(f"no row count gives {regime} for K={K} L={L} on {sms} SMs")


@pytest.mark.parametrize("K,model,sd,regime", _dw_cases())
def test_weight_gradients_exact(K, model, sd, regime):
    """mmf_pf_heads_weight_grads on small-integer inputs equals float64 bit for bit (dW, db, g_in, g_out), with the
    reference missing one row as a negative control."""
    sms = _sms()
    L = _head_depth(model)
    P = find_rows(K, L, regime, sms)
    q = dw_regime(K, L, P, sms)
    if regime == "c4":
        assert P == 245760 and q["chunks"] >= 2 and q["tiles_per_chunk"] >= 4, q
    elif regime.startswith("P"):
        assert P < DWT_ROWS and q["chunks"] == 1 and q["ragged"], q
    else:
        t = int(regime.split()[0])
        assert q["chunks"] >= 2 and q["tiles_per_chunk"] == t, q
        assert q["last_chunk_rows"] == 1 if regime.endswith("1 row") else (q["ragged"] and q["last_chunk_tiles"] == t), q
    g = torch.Generator(device=DEV).manual_seed(1000 * K + P)
    ints = lambda *shape: torch.randint(-2, 3, shape, device=DEV, generator=g).float()  # noqa: E731
    act, delta = ints(K, L + 1, U // 4, P, 4), ints(K, L + 1, U // 4, P, 4)
    x, d_ll = ints(P, sd), ints(K, P)
    x[P - 1], d_ll[:, P - 1] = 1.0, 2.0  # the control row below contributes to every output
    dW, db, g_in, g_out = profiled(lambda: weight_grads(act, delta, x, d_ll), DW)
    A, D = ops.rows_view(act).double(), ops.rows_view(delta).double()  # (K, L + 1, P, 64)
    xd, dd = x.double(), d_ll.double()

    def reference(rows):
        a, d, xs, w = A[:, :, rows], D[:, :, rows], xd[rows], dd[:, rows]
        return (torch.einsum("klpi,klpj->klij", d[:, :L], a[:, :L]), d.sum(dim=2),
                torch.einsum("kpi,pd->kid", d[:, L], xs), torch.einsum("kpi,kp->ki", a[:, L], w))

    got = [t.double() for t in (dW, db, g_in, g_out)]
    names = ("dW", "db", "g_in", "g_out")
    ref = reference(slice(None))
    for name, a, e in zip(names, got, ref):
        assert torch.equal(a, e), (f"{name}: {int((a != e).sum())} entries differ, worst "
                                   f"{float(torch.nan_to_num((a - e).abs(), nan=math.inf).max())}")
    # negative control: the same comparison sees the last row dropped from the reference, or counted twice
    last = reference(slice(P - 1, P))
    for sign in (-1.0, 1.0):
        for name, a, e, c in zip(names, got, ref, last):
            assert not torch.equal(a, e + sign * c), f"{name}: a one-row change of the reference goes unseen"


# ---- the whole training step ----------------------------------------------------------------------------------------
def bptt(side, precision, T, N, Mp, seed, dtype=torch.float32, dev=DEV):
    name, sd = "PushCrossmodalParticleFilter", 2
    init, eps, _ = draw_noise(T, N, Mp, sd, seed=seed)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=seed + 1)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd)
    if side == "oracle":
        f = fill_parameters(getattr(port, name)(), seed=47).to(device=dev, dtype=dtype)
        f.noise = RecordedNoise(init_eps=init, process_eps=eps)
    else:
        f = fill_parameters(M.PushCrossmodalParticleFilter(), seed=47).to(DEV)
        f.noise = ReplayNoise(init_eps=init, process_eps=eps)
        f.precision = precision
    f.train()
    f.num_particles = Mp
    for prm in f.dynamics_model.parameters():
        prm.requires_grad_(False)
    cvt = lambda t: t.to(device=dev, dtype=dtype)  # noqa: E731
    f.initialize_beliefs(mean=cvt(states[0]), covariance=cvt(cov).contiguous())
    est = f.forward_loop(observations={k: cvt(v[1:]) for k, v in obs.items()}, controls=cvt(controls[1:]))
    loss = torch.mean((est - cvt(states[1:])) ** 2)
    loss.backward()
    return loss.item(), {k: q.grad.detach().double().cpu() for k, q in f.named_parameters() if q.grad is not None}


def gradient_report(go, gp):
    """(relative L2, cosine, tensor) of every parameter gradient that carries gradient mass (>= 1e-4 of the largest
    norm): a ReLU that flips between the two evaluations changes one particle's contribution below it by O(1), so the
    comparison is per tensor (direction and magnitude) rather than per entry."""
    assert set(go) == set(gp) and len(go) > 50
    big = max(float(g.norm()) for g in go.values())
    report = []
    for k in go:
        ref, got = go[k].reshape(-1), gp[k].reshape(-1)
        if float(ref.norm()) < 1e-4 * big:
            continue
        report.append((float((ref - got).norm() / ref.norm()), float(torch.dot(ref, got) / (ref.norm() * got.norm())), k))
    return sorted(report, reverse=True)




def test_c4_training_step_against_float64_oracle():
    """The fused bf16x3 training step (FusedHeads, Reweight, HeadGradToken, the d_rows sum) at C4's batch, N = 8192 x
    M = 30, frozen dynamics, against the oracle port in float64 on the GPU, over T = 2 filter steps (the gradient crosses a
    step through the log-weights): the float64 reference keeps every activation of the particle chains and image
    encoders for the backward, 18 GiB per step at this batch (peak 37.7 GiB at T = 2, 55.3 GiB at T = 3, measured on a
    B200), so T = 15 would take ~280 GiB.  Bars: those of test_c4_gradients_at_15_steps (loss 1e-4 relative; per tensor
    relative L2 <= 5e-3 and cosine >= 0.99999), kept: measured on a B200, loss 1.1e-7, worst relative L2 8.7e-4 and
    lowest cosine 0.9999996 (the first convolution of the image encoder).  A second identical run must give
    bit-identical gradients (cuDNN deterministic for the encoders' convolutions, which are outside this library)."""
    T, N, Mp, seed = 2, C4_N, C4_M, 81
    t0 = time.time()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    lo, go = bptt("oracle", None, T, N, Mp, seed, dtype=torch.float64)
    torch.cuda.synchronize()
    peak = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
    t1 = time.time()
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        runs = []
        for _ in range(2):
            ops.PROFILE.reset(enabled=True)
            runs.append(bptt("product", "bf16x3", T, N, Mp, seed))
            prof = ops.PROFILE.collect()
            ops.PROFILE.reset()
            for entry in ("pf_heads_forward_train", "pf_heads_backward", "pf_heads_weight_grads"):
                assert prof["kernels"].get(entry, {}).get("count") == T, f"{entry} did not run once per step: {prof['kernels']}"
    finally:
        torch.backends.cudnn.deterministic = det
    (lp, gp), (lp2, gp2) = runs
    report = gradient_report(go, gp)
    print(f"[c4 N={N} T={T}] float64 reference: peak {peak:.1f} GiB, {t1 - t0:.1f} s; loss {lp:.8f} vs {lo:.8f} "
          f"(rel {abs(lp - lo) / abs(lo):.2e}); worst (rel L2, cos, tensor): {report[:4]}")
    assert abs(lp - lo) <= 1e-4 * abs(lo)
    assert all(rel <= 5e-3 and cos >= 0.99999 for rel, cos, _ in report), f"worst (rel L2, cos, tensor): {report[:5]}"
    differing = [k for k in gp if not torch.equal(gp[k], gp2[k])]
    assert lp == lp2 and not differing, f"gradients differ between two identical runs: {differing[:5]}"


# ---- single-pass bf16 training --------------------------------------------------------------------------------------
# measured on a B200: loss 1.0e-4 relative, worst tensor relative L2 0.043, lowest cosine 0.99908 (both on the first
# convolution of the image encoder); bars at 10x, 2.3x and 5x (in 1 - cos) of that
BF16_LOSS, BF16_REL, BF16_COS = 1e-3, 0.1, 0.995


def test_bf16_training_gradients_against_oracle():
    """precision = "bf16" (forward on the hi halves of the split operands only, backward with the three split MMAs) at
    the C4-mini shape (N = 48, M = 30, T = 15) against the fp32 oracle, flip-aware per tensor."""
    T, N, Mp, seed = 15, 48, 30, 45
    lo, go = bptt("oracle", None, T, N, Mp, seed, dev="cpu")
    ops.PROFILE.reset(enabled=True)
    lb, gb = bptt("product", "bf16", T, N, Mp, seed)
    prof = ops.PROFILE.collect()
    ops.PROFILE.reset()
    assert prof["kernels"].get("pf_heads_forward_train", {}).get("count") == T, prof["kernels"]
    report = gradient_report(go, gb)
    print(f"[bf16 N={N} T={T}] loss {lb:.6f} vs {lo:.6f} (rel {abs(lb - lo) / abs(lo):.2e}); "
          f"worst (rel L2, cos, tensor): {report[:4]}; best cos {min(r[1] for r in report):.6f}")
    assert abs(lb - lo) <= BF16_LOSS * abs(lo)
    assert all(rel <= BF16_REL and cos >= BF16_COS for rel, cos, _ in report), f"worst (rel L2, cos, tensor): {report[:5]}"
