"""The Kalman-filter kernels and the dynamics rollout at the sizes where their persistent loops run (the Kalman
train_filter step and eval at N = 4096 trajectories, T = 100 steps of eval: 409,600 fused rows), against float64.

    k_ekf_loop<SD,TAPE>       a warp per (filter, trajectory) for all T steps; wpc = clamp(ceil(F N / SMs), 1, 16) warps
                              per CTA, fewer while the packed chain and the per-warp scratch overflow the shared-memory
                              window; grid (min(ceil(N / wpc), SMs / F), F); a warp takes trajectory n + ctas wpc next,
                              reusing its registers and shared scratch.  jac_only (mmf_dynamics_jacobian): F = 1, T = 1
    k_ekf_loop_bwd<SD>        a thread per (filter, trajectory), at most 148 x 16 blocks of 128: 303,104 items a round
    k_kf_fuse<SD>             R10 / R11, a thread per row, the same 303,104-row rounds
    k_kf_fuse_measurements    R12, the same
    k_dyn_rollout<SD,TAPE>    a warp per trajectory; wpc = clamp(ceil(N / SMs), 1, 32), fewer to fit; min(ceil(N / wpc),
                              SMs) CTAs

Every case restates its launcher's arithmetic in Python and asserts before it runs that it is in the intended regime (two
rounds or more, a ragged last round); test_regimes_of_the_shapes checks those restatements at a B200's 148 SMs and
232,448-byte window without a device.  torch.profiler confirms the kernel that ran; outputs are NaN-prefilled and the
kernels are called through the raw C entry points, so an element never written fails.  References are float64 on the GPU
in chunks of at most 2^18 rows, compared per row (worst |got - ref| / max(|ref|, rms(ref)), reported with its
(filter, step, trajectory)):

  * EKF: teacher-forced per step.  From the kernel's own posterior of step t-1 (mean0 / cov0 at t = 0): the hoisted
    control row, mu- = f(mu) and A = df/dx (torch.func.jacfwd) through the float64 chain, then Pp = A P A^T + Q Q^T,
    S = Pp + R R^T, K = Pp S^-1, mu = mu- + K (z - mu-), P = (I - K) Pp.  The recursion amplifies rounding on some
    trajectories; teacher forcing removes that and still shows a misplaced trajectory, step, filter or round as O(1);
  * EKF backward: float64 autograd through the recursion fed the kernel's tape (A and mu- of every step);
  * R10 / R11 / R12: the formulas of include/mmf_b200.h and the reference expressions (models._information_fusion,
    models._measurement_level) in float64;
  * rollout: teacher-forced, x_{t+1} through the float64 chain from the kernel's own x_t; every tape plane against the
    float64 input of its layer there.

Bars start from the neighbouring tests'.  A wrong trajectory, round or filter is wrong by O(1).
"""
import ctypes as C

import pytest
import torch

from multimodalfilter_b200 import _lib, fused, ops
from multimodalfilter_b200.crossmodal import models as M
from multimodalfilter_b200.synthetic import fill_parameters

from full_size import assert_rows, chain_forward, profiled, row_excess

DEV = "cuda:0"
U = _lib.UNITS
f64 = torch.float64
CHUNK = 1 << 18              # rows per float64 reference chunk
B200_SMS, B200_WINDOW = 148, 232448
EKF_MAX_WARPS, DYN_MAX_WARPS = 16, 32
FLAT_ROUND = 148 * 16 * 128  # k_ekf_loop_bwd, k_kf_fuse, k_kf_fuse_measurements: items per grid-stride round
RTOL_MEAN = 2e-5             # means, mu-, rollout states
RTOL_COV = 1e-4              # covariances, A
RTOL_PLANES = 2e-5           # tape planes (RTOL_ROWS of the inference tests)
RTOL_BWD = 2e-4
KINK = 1e-5                  # dynamics64: a pre-activation this close to zero (relative) may flip sides in fp32
RTOL_R10, RTOL_R11, RTOL_R12_Z, RTOL_R12_COV = 1e-5, 1e-4, 1e-5, 1e-4
RTOL_R12_FACTOR = 1e-5
RTOL_R12_QUIRK = 4e-3        # unimodal K > 1, sd = 4: fp32 Gauss-Jordan of a matrix holding K 1e9 above its diagonal
KAPPA_FACTOR = 8             # R11 at kappa > 1e2 and the R12 factor: per-row bar KAPPA_FACTOR cond 2^-24


# ---- the launchers' arithmetic, restated ----------------------------------------------------------------------------
def _rounds(items, per_round):
    rounds = -(-items // per_round)
    return {"per_round": per_round, "rounds": rounds, "last_round": items - per_round * (rounds - 1)}


def ekf_regime(F, sd, N, nf, sms, window):
    """launch_ekf_sd: warps per CTA, CTAs per filter, trajectories per round of one filter."""
    warp_floats = 3 * (1 + sd) * U + 384
    wpc = max(1, min(EKF_MAX_WARPS, -(-F * N // sms)))
    while (((nf + 3) & ~3) + wpc * warp_floats) * 4 > window and wpc > 1:
        wpc -= 1
    ctas = min(-(-N // wpc), max(sms // F, 1))
    return {"wpc": wpc, "ctas": ctas, **_rounds(N, ctas * wpc)}


def dyn_regime(N, nf, sms, window):
    """launch_dyn_rollout_sd / dyn_launch_shape."""
    wpc = max(1, min(DYN_MAX_WARPS, -(-N // sms)))
    while (((nf + 3) & ~3) + wpc * (3 * U + 384)) * 4 > window and wpc > 1:
        wpc -= 1
    ctas = min(-(-N // wpc), sms)
    return {"wpc": wpc, "ctas": ctas, **_rounds(N, ctas * wpc)}


def flat_regime(items):
    return _rounds(items, FLAT_ROUND)


def _device():
    p = torch.cuda.get_device_properties(0)
    return p.multi_processor_count, p.shared_memory_per_block_optin


def _assert_loops(g, loops=True):
    if loops:
        assert g["rounds"] >= 2 and 0 < g["last_round"] < g["per_round"], g
    else:
        assert g["rounds"] == 1, g


# ---- the shapes ------------------------------------------------------------------------------------------------------
# (id, F, sd, N, T, regime at 148 SMs and a 232,448-byte window)
EKF_CASES = [
    ("kalman_train", 2, 3, 4096, 15, dict(wpc=16, ctas=74, rounds=4, last_round=544)),
    ("kalman_eval", 2, 3, 4096, 100, dict(wpc=16, ctas=74, rounds=4, last_round=544)),
    ("push", 2, 2, 2 * 1184 + 3, 15, dict(wpc=16, ctas=74, rounds=3, last_round=3)),
    ("one_filter", 1, 3, 2 * 2368 + 37, 15, dict(wpc=16, ctas=148, rounds=3, last_round=37)),
    ("three_filters", 3, 1, 3 * 784 + 5, 15, dict(wpc=16, ctas=49, rounds=4, last_round=5)),
    ("four_filters_sd4", 4, 4, 2 * 518 + 1, 15, dict(wpc=14, ctas=37, rounds=3, last_round=1)),
    ("c2_control", 2, 3, 256, 100, dict(wpc=4, ctas=64, rounds=1, last_round=256)),
]
JAC_CASES = [(sd, N) for sd in (2, 3) for N in (2 * 2368 + 5, 4096)]
JAC_REGIMES = {2 * 2368 + 5: dict(wpc=16, ctas=148, rounds=3, last_round=5),
               4096: dict(wpc=16, ctas=148, rounds=2, last_round=1728)}
# (id, F, sd, N, T, rounds of 303,104 items, items of the last round)
BWD_CASES = [("one_filter", 1, 3, 2 * FLAT_ROUND + 37, 3, 3, 37), ("two_filters_sd4", 2, 4, 151571, 4, 2, 38)]
FUSE_ROWS = [409600, 2 * FLAT_ROUND + 3]
FUSE_REGIMES = {409600: (2, 409600 - FLAT_ROUND), 2 * FLAT_ROUND + 3: (3, 3)}
FUSE_KSD = [(2, 3), (2, 2), (1, 3), (3, 4), (4, 1)]
DYN_N = 3 * 4736 + 5
DYN_REGIME = dict(wpc=32, ctas=148, rounds=4, last_round=5)


def _dyn_class(sd):
    """Push (sd 2) and Door (sd 3) dynamics, or the door layout with another state width."""
    if sd == 2:
        return M.PushDynamicsModel
    if sd == 3:
        return M.DoorDynamicsModel
    return type(f"Dyn{sd}", (M._Dynamics,), {"_STATE_DIM": sd, "_NOISE": ("tril", [0.05, 0.01, 0.01, 0.02][:sd], 1.0)})


def _nf(sd):
    """Floats of the packed state chain (EKFPlan._buffers[2 f]) of a dynamics model of state width sd."""
    return fused._DynamicsSpec(_dyn_class(sd)()).pack()[0].numel()


def test_regimes_of_the_shapes():
    """The restated launch arithmetic at 148 SMs and the 232,448-byte window puts every shape of this file in the regime
    it is meant for; sd = 4 at 16 warps would need more than the window, so the launcher takes 14."""
    sms, win = B200_SMS, B200_WINDOW
    for name, F, sd, N, _, want in EKF_CASES:
        g = ekf_regime(F, sd, N, _nf(sd), sms, win)
        assert {k: g[k] for k in want} == want, (name, g)
        _assert_loops(g, loops=name != "c2_control")
    assert ((_nf(4) + 3) & ~3) * 4 + 16 * (3 * 5 * U + 384) * 4 > win >= ((_nf(4) + 3) & ~3) * 4 + 14 * (3 * 5 * U + 384) * 4
    for sd, N in JAC_CASES:
        g = ekf_regime(1, sd, N, _nf(sd), sms, win)
        assert {k: g[k] for k in JAC_REGIMES[N]} == JAC_REGIMES[N], (sd, N, g)
    for name, F, sd, N, T, rounds, last in BWD_CASES:
        g = flat_regime(F * N)
        assert (g["rounds"], g["last_round"]) == (rounds, last), (name, g)
        assert ekf_regime(F, sd, N, _nf(sd), sms, win)["rounds"] >= 2, name
    assert FLAT_ROUND // 151571 == 1, "the second round of the two-filter case lies in filter 1"
    for rows in FUSE_ROWS:
        g = flat_regime(rows)
        assert (g["rounds"], g["last_round"]) == FUSE_REGIMES[rows], (rows, g)
    for sd in (1, 2, 3, 4):
        g = dyn_regime(DYN_N, _nf(sd), sms, win)
        assert {k: g[k] for k in DYN_REGIME} == DYN_REGIME, (sd, g)


# ---- models and raw entry points -----------------------------------------------------------------------------------
def _ekf_plan(F, sd, seed):
    """F dynamics of state width sd, each with its own weights and its own lower-triangular process-noise factor
    (fill_parameters leaves Q_scale_tril at the class's constant, which would make every filter's Q the same)."""
    filters = []
    for f in range(F):
        dyn = fill_parameters(_dyn_class(sd)(), seed=seed + f).to(DEV)
        g = torch.Generator().manual_seed(seed + 100 * f)
        q = torch.tril(0.05 * torch.randn(sd, sd, generator=g), -1) + torch.diag(0.1 + 0.2 * torch.rand(sd, generator=g))
        with torch.no_grad():
            dyn.Q_scale_tril.copy_(q * (1 + f))
        for p in dyn.parameters():
            p.requires_grad_(False)
        filters.append(type("H", (), {"dynamics_model": dyn})())
    plan = fused.EKFPlan.build(filters)
    assert plan is not None
    plan.refresh(torch.device(DEV))
    return plan


def _plan_nf(plan):
    return max(plan._buffers[2 * f].numel() for f in range(len(plan.dyns)))


def _ekf_inputs(F, T, N, sd, seed):
    """mean0, cov0 = 0.1 I, controls, z, R with diagonal >= 0.1 (test_ekf_training._inputs)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    mean0 = torch.randn(F, N, sd, device=DEV, generator=g)
    cov0 = (0.1 * torch.eye(sd, device=DEV)).expand(F, N, sd, sd).contiguous()
    z = torch.randn(F, T, N, sd, device=DEV, generator=g)
    R = torch.tril(0.05 * torch.randn(F, T, N, sd, sd, device=DEV, generator=g))
    R = R + torch.diag_embed(0.1 + torch.rand(F, T, N, sd, device=DEV, generator=g))
    u = torch.randn(T, N, 7, device=DEV, generator=g)
    return mean0, cov0, u, z, R


def _nan(*shape):
    return torch.full(shape, float("nan"), device=DEV)


def ekf_raw(plan, mean0, cov0, u, z, R, tape):
    F, T, N, sd = z.shape
    means, covs = _nan(F, T, N, sd), _nan(F, T, N, sd, sd)
    arr = (_lib.EKFModel * F)(*plan.structs)
    lib = _lib.load()
    args = [_lib.ptr(x) for x in (mean0, cov0, u, z, R, means, covs)]
    if not tape:
        _lib.check(_lib.call(lib.mmf_ekf_loop_fwd, arr, F, T, N, *args, _lib.stream_of(z)))
        return means, covs
    pred, jac = _nan(F, T, N, sd), _nan(F, T, N, sd, sd)
    _lib.check(_lib.call(lib.mmf_ekf_loop_train_fwd, arr, F, T, N, *args, _lib.ptr(pred), _lib.ptr(jac),
                         _lib.stream_of(z)))
    return means, covs, pred, jac


def jacobian_raw(plan, states, controls):
    N, sd = states.shape
    pred, jac = _nan(N, sd), _nan(N, sd, sd)
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_dynamics_jacobian, C.byref(plan.structs[0]), N, _lib.ptr(states), _lib.ptr(controls),
                         _lib.ptr(pred), _lib.ptr(jac), _lib.stream_of(states)))
    return pred, jac


def ekf_bwd_raw(plan, cov0, z, R, covs, pred, jac, d_means, d_covs):
    F, T, N, sd = z.shape
    outs = [_nan(F, N, sd), _nan(F, N, sd, sd), _nan(F, T, N, sd), _nan(F, T, N, sd, sd)]
    arr = (_lib.EKFModel * F)(*plan.structs)
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_ekf_loop_bwd, arr, F, T, N, None, _lib.ptr(cov0), _lib.ptr(z), _lib.ptr(R), None,
                         _lib.ptr(covs), _lib.ptr(pred), _lib.ptr(jac), _lib.ptr(d_means), _lib.ptr(d_covs),
                         *[_lib.ptr(o) for o in outs], _lib.stream_of(z)))
    return outs


def _q64(plan, f):
    sd = plan.sd
    q = torch.tensor(list(plan.structs[f].q_tril)[:sd * sd], dtype=f64, device=DEV).reshape(sd, sd)
    return q @ q.T


def _labels(*dims):
    """Row -> 'f=.. t=.. n=..' for rows enumerated over dims = (("f", F), ("t", T), ("n", N)) ..."""
    def where(row):
        parts = []
        for name, size in reversed(dims):
            parts.append(f"{name}={row % size}")
            row //= size
        return " ".join(reversed(parts))
    return where


# ---- float64 dynamics -------------------------------------------------------------------------------------------------
def control_rows64(spec, u):
    """The hoisted mid-layer rows of controls u (P, cd): the control encoder, then the mid Linear's control columns and
    bias (fused.pack_rows), in float64."""
    d = lambda t: t.detach().double()  # noqa: E731
    enc_lin, enc_res = spec.control
    h = torch.relu(u.double() @ d(enc_lin.weight).T + d(enc_lin.bias))
    for r in enc_res:
        t = torch.relu(h @ d(r.block1.weight).T + d(r.block1.bias))
        h = torch.relu(t @ d(r.block2.weight).T + d(r.block2.bias) + h)
    mid = spec.shared[0]
    return h @ d(mid.weight[:, :U]).T + d(mid.bias)


def dynamics64(spec, x, rb, jacobian=False, planes=None):
    """f(x) = x + y[:sd] sigmoid(y[sd]) through the float64 chain on rows x (P, sd), rows rb (P, 64); with `jacobian`
    also A = df/dx (P, sd, sd) by torch.func.jacfwd and the rows at a ReLU kink (P,) bool: some unit's pre-activation
    within KINK of zero (relative to the rms of its layer's), where fp32 and float64 may take different sides and A
    jumps by that unit's whole contribution."""
    sd = spec.sd
    x = x.double()

    def f(v, planes=None, preacts=None):
        xv = x + v
        y = chain_forward(spec.state, spec.shared, slice(U, 2 * U), xv, rb, mid_relu=False, planes=planes,
                          preacts=preacts)
        return xv + y[:, :sd] * torch.sigmoid(y[:, sd:sd + 1])

    v0 = torch.zeros(sd, dtype=f64, device=x.device)
    preacts = []
    fx = f(v0, planes, preacts)
    if not jacobian:
        return fx
    kink = torch.zeros(x.shape[0], dtype=torch.bool, device=x.device)
    for a in preacts:
        kink |= (a.abs() < KINK * a.pow(2).mean(1, keepdim=True).sqrt()).any(1)
    return fx, torch.func.jacfwd(f)(v0), kink


def ekf_teacher_forced(plan, mean0, cov0, u, z, R, means, covs):
    """The float64 step of every (f, t, n) from the kernel's own posterior of step t-1: mu-, A, mu, P (F, T N, ...) and
    the steps at a ReLU kink (F, T N)."""
    F, T, N, sd = z.shape
    TN = T * N
    out = [torch.empty(F, TN, sd, dtype=f64, device=DEV), torch.empty(F, TN, sd, sd, dtype=f64, device=DEV),
           torch.empty(F, TN, sd, dtype=f64, device=DEV), torch.empty(F, TN, sd, sd, dtype=f64, device=DEV),
           torch.empty(F, TN, dtype=torch.bool, device=DEV)]
    eye = torch.eye(sd, dtype=f64, device=DEV)
    uu = u.reshape(TN, -1)
    for f in range(F):
        spec, Q = plan.dyns[f], _q64(plan, f)
        mu_prev = torch.cat([mean0[f][None], means[f, :-1]]).reshape(TN, sd)
        P_prev = torch.cat([cov0[f][None], covs[f, :-1]]).reshape(TN, sd, sd)
        zz, RR = z[f].reshape(TN, sd).double(), R[f].reshape(TN, sd, sd).double()
        for a in range(0, TN, CHUNK):
            b = min(TN, a + CHUNK)
            pred, A, out[4][f, a:b] = dynamics64(spec, mu_prev[a:b], control_rows64(spec, uu[a:b]), jacobian=True)
            Pp = A @ P_prev[a:b].double() @ A.mT + Q
            S = Pp + RR[a:b] @ RR[a:b].mT
            K = torch.linalg.solve(S.mT, Pp.mT).mT  # Pp S^-1
            out[0][f, a:b], out[1][f, a:b] = pred, A
            out[2][f, a:b] = pred + (K @ (zz[a:b] - pred)[..., None])[..., 0]
            out[3][f, a:b] = (eye - K) @ Pp
    return out


def _smooth(kink):
    """Indices of the rows away from every ReLU kink; the kinks must stay rare, or the check would thin out."""
    assert float(kink.float().mean()) < 0.01, f"{int(kink.sum())} of {kink.numel()} rows at a ReLU kink"
    return (~kink).nonzero()[:, 0]


def assert_kept(got, ref, keep, bar, what, report, category, where):
    """assert_rows on the rows `keep`, reported by their own labels."""
    assert_rows(got[keep], ref[keep], bar, what, report, category, lambda row: where(int(keep[row])))


# ---- a. k_ekf_loop, eval and tape ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", EKF_CASES, ids=[c[0] for c in EKF_CASES])
def test_ekf_loop_matches_float64_teacher_forced(case):
    """mmf_ekf_loop_fwd and mmf_ekf_loop_train_fwd past one round of trajectories: posteriors of every (f, t, n), and
    the tape's mu- and A, against the float64 step from the kernel's own previous posterior; eval and tape forward agree
    bit for bit."""
    name, F, sd, N, T, _ = case
    plan = _ekf_plan(F, sd, seed=10 + sd)
    regime = ekf_regime(F, sd, N, _plan_nf(plan), *_device())
    _assert_loops(regime, loops=name != "c2_control")
    mean0, cov0, u, z, R = _ekf_inputs(F, T, N, sd, seed=N + T)
    means, covs = profiled(lambda: ekf_raw(plan, mean0, cov0, u, z, R, tape=False), [f"k_ekf_loop<{sd},false>"])
    tm, tc, pred, jac = profiled(lambda: ekf_raw(plan, mean0, cov0, u, z, R, tape=True), [f"k_ekf_loop<{sd},true>"])
    assert torch.equal(means, tm) and torch.equal(covs, tc), "eval and tape forward differ"
    pred_ref, A_ref, mean_ref, cov_ref, kink = ekf_teacher_forced(plan, mean0, cov0, u, z, R, means, covs)
    rows, where, report = F * T * N, _labels(("f", F), ("t", T), ("n", N)), {}
    keep = _smooth(kink.reshape(rows))
    assert_rows(pred.reshape(rows, sd), pred_ref.reshape(rows, sd), RTOL_MEAN, "pred_out", report, "pred", where)
    assert_kept(jac.reshape(rows, -1), A_ref.reshape(rows, -1), keep, RTOL_COV, "jac_out", report, "A", where)
    assert_kept(means.reshape(rows, sd), mean_ref.reshape(rows, sd), keep, RTOL_MEAN, "mean_out", report, "mean", where)
    assert_kept(covs.reshape(rows, -1), cov_ref.reshape(rows, -1), keep, RTOL_COV, "cov_out", report, "cov", where)
    print(f"[{name}] F={F} sd={sd} N={N} T={T} {regime}; {rows - keep.numel()} of {rows} steps at a kink; worst "
          "relative errors " + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- b. mmf_dynamics_jacobian ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sd,N", JAC_CASES)
def test_dynamics_jacobian_matches_float64(sd, N):
    """The jac_only path of k_ekf_loop past one round: f and df/dx at given states against float64."""
    plan = _ekf_plan(1, sd, seed=30 + sd)
    regime = ekf_regime(1, sd, N, _plan_nf(plan), *_device())
    _assert_loops(regime)
    g = torch.Generator(device=DEV).manual_seed(N + sd)
    states = torch.randn(N, sd, device=DEV, generator=g)
    controls = torch.randn(N, 7, device=DEV, generator=g)
    pred, jac = profiled(lambda: jacobian_raw(plan, states, controls), [f"k_ekf_loop<{sd},false>"])
    spec = plan.dyns[0]
    pred_ref, A_ref, kink = dynamics64(spec, states, control_rows64(spec, controls), jacobian=True)
    report, where = {}, _labels(("n", N))
    keep = _smooth(kink)
    assert_rows(pred, pred_ref, RTOL_MEAN, "pred", report, "pred", where)
    assert_kept(jac.reshape(N, -1), A_ref.reshape(N, -1), keep, RTOL_COV, "jacobian", report, "A", where)
    print(f"[sd={sd} N={N}] {regime}; {N - keep.numel()} states at a kink; worst relative errors "
          + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- c. k_ekf_loop_bwd beyond one round ------------------------------------------------------------------------------
def tape_fed_grads(plan, mean0, cov0, z, R, pred, jac, d_means, d_covs):
    """float64 autograd through the recursion fed the tape: mu-_t = pred_t + A_t (mu_{t-1} - mu_{t-1}.detach()) (the
    tape's value, derivative A_t).  -> d_mean0, d_cov0, d_z, d_r_tril."""
    F, T, N, sd = z.shape
    Q = torch.stack([_q64(plan, f) for f in range(F)])[:, None]
    m0, P0, zz, RR = (x.double().requires_grad_(True) for x in (mean0, cov0, z, R))
    A, pr = jac.double(), pred.double()
    eye = torch.eye(sd, dtype=f64, device=DEV)
    mu, P, loss = m0, P0, 0.0
    for t in range(T):
        mp = pr[:, t] + (A[:, t] @ (mu - mu.detach())[..., None])[..., 0]
        Pp = A[:, t] @ P @ A[:, t].mT + Q
        S = Pp + RR[:, t] @ RR[:, t].mT
        K = torch.linalg.solve(S.mT, Pp.mT).mT
        mu = mp + (K @ (zz[:, t] - mp)[..., None])[..., 0]
        P = (eye - K) @ Pp
        loss = loss + (mu * d_means[:, t].double()).sum()
        if d_covs is not None:
            loss = loss + (P * d_covs[:, t].double()).sum()
    return torch.autograd.grad(loss, (m0, P0, zz, RR))


@pytest.mark.gpu
@pytest.mark.parametrize("case", BWD_CASES, ids=[c[0] for c in BWD_CASES])
@pytest.mark.parametrize("with_d_covs", [True, False])
def test_ekf_loop_bwd_matches_float64_given_the_tape(case, with_d_covs):
    """mmf_ekf_loop_bwd past 303,104 (filter, trajectory) items, fed the tape of mmf_ekf_loop_train_fwd: d_mean0 and
    d_cov0 of every (f, n), d_z and d_r_tril of every (f, t, n) against float64 autograd, per row."""
    name, F, sd, N, T, _, _ = case
    regime = flat_regime(F * N)
    _assert_loops(regime)
    plan = _ekf_plan(F, sd, seed=40 + sd)
    mean0, cov0, u, z, R = _ekf_inputs(F, T, N, sd, seed=N + T)
    _, covs, pred, jac = ekf_raw(plan, mean0, cov0, u, z, R, tape=True)
    g = torch.Generator(device=DEV).manual_seed(F * N)
    d_means = torch.randn(F, T, N, sd, device=DEV, generator=g)
    d_covs = torch.randn(F, T, N, sd, sd, device=DEV, generator=g) if with_d_covs else None
    got = profiled(lambda: ekf_bwd_raw(plan, cov0, z, R, covs, pred, jac, d_means, d_covs), [f"k_ekf_loop_bwd<{sd}>"])
    want = tape_fed_grads(plan, mean0, cov0, z, R, pred, jac, d_means, d_covs)
    report = {}
    fn, ftn = _labels(("f", F), ("n", N)), _labels(("f", F), ("t", T), ("n", N))
    for what, a, b, rows, where in zip(("d_mean0", "d_cov0", "d_z", "d_r_tril"), got, want,
                                       (F * N, F * N, F * T * N, F * T * N), (fn, fn, ftn, ftn)):
        assert_rows(a.reshape(rows, -1), b.reshape(rows, -1), RTOL_BWD, what, report, what, where)
    print(f"[{name} d_covs={'given' if with_d_covs else 'NULL'}] F={F} sd={sd} N={N} T={T} {regime}; worst relative "
          "errors " + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- d. R10 / R11 k_kf_fuse and R12 k_kf_fuse_measurements past 303,104 rows --------------------------------------
def fuse_raw(K, rows, sd, mu, P, beta):
    mean, cov = _nan(rows, sd), _nan(rows, sd, sd)
    lib = _lib.load()
    if beta is None:
        _lib.check(_lib.call(lib.mmf_kf_fuse_unimodal, K, rows, sd, _lib.ptr(mu), _lib.ptr(P), _lib.ptr(mean),
                             _lib.ptr(cov), _lib.stream_of(mu)))
    else:
        _lib.check(_lib.call(lib.mmf_kf_fuse_crossmodal, K, rows, sd, _lib.ptr(mu), _lib.ptr(P), _lib.ptr(beta),
                             _lib.ptr(mean), _lib.ptr(cov), _lib.stream_of(mu)))
    return mean, cov


def fuse_measurements_raw(K, rows, sd, z, tril, w):
    z_out, mat = _nan(rows, sd), _nan(rows, sd, sd)
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_kf_fuse_measurements, K, rows, sd, _lib.ptr(z), _lib.ptr(tril), _lib.ptr(w),
                         _lib.ptr(z_out), _lib.ptr(mat), _lib.stream_of(z)))
    return z_out, mat


def _fuse_regime(rows):
    regime = flat_regime(rows)
    _assert_loops(regime)
    return regime


def _spd(K, rows, sd, kappa, g):
    """SPD matrices V diag(lam) V^T (V a Householder reflection) with condition number <= kappa by construction, and
    that condition number per (k, row)."""
    v = torch.randn(K, rows, sd, 1, dtype=f64, device=DEV, generator=g)
    V = torch.eye(sd, dtype=f64, device=DEV) - 2 * v @ v.mT / (v.mT @ v)
    scale = 10 ** (torch.rand(K, rows, 1, dtype=f64, device=DEV, generator=g) - 0.5)
    lam = scale * kappa ** -torch.rand(K, rows, sd, dtype=f64, device=DEV, generator=g)
    P = (V * lam[..., None, :]) @ V.mT
    return P.float().contiguous(), lam.amax(-1) / lam.amin(-1)


@pytest.mark.gpu
@pytest.mark.parametrize("rows", FUSE_ROWS)
@pytest.mark.parametrize("K,sd", FUSE_KSD)
def test_kf_fuse_crossmodal_matches_float64(K, sd, rows):
    """R10 (mmf_kf_fuse_crossmodal): mean = sum_k beta_k / (sum beta + 1e-9) mu_k, cov = sum_k beta_k beta_k^T o P_k
    (CrossmodalKalmanFilter.calculate_weighted_states) in float64, with one modality blacked out (beta 0) on a fifth of
    the rows and every beta 0 on a few (mean 0 there)."""
    regime = _fuse_regime(rows)
    g = torch.Generator(device=DEV).manual_seed(rows + 10 * K + sd)
    mu = torch.randn(K, rows, sd, device=DEV, generator=g)
    P, _ = _spd(K, rows, sd, 1e2, g)
    beta = 1.0 - torch.rand(K, rows, sd, device=DEV, generator=g)  # (0, 1]
    if K > 1:
        beta[0, ::5] = 0.0
    beta[:, 1::9973] = 0.0
    mean, cov = profiled(lambda: fuse_raw(K, rows, sd, mu, P, beta), [f"k_kf_fuse<{sd}>"])
    b = beta.double()
    mean_ref = (b / (b.sum(0) + 1e-9) * mu.double()).sum(0)
    cov_ref = ((b[..., :, None] * b[..., None, :]) * P.double()).sum(0)
    assert not mean_ref[1::9973].any()
    report, where = {}, _labels(("row", rows))
    assert_rows(mean, mean_ref, RTOL_R10, "mean", report, "mean", where)
    assert_rows(cov.reshape(rows, -1), cov_ref.reshape(rows, -1), RTOL_R10, "cov", report, "cov", where)
    print(f"[K={K} sd={sd} rows={rows}] {regime}; worst relative errors "
          + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("rows,K,sd,kappa", [(r, K, sd, 1e2) for r in FUSE_ROWS for K, sd in FUSE_KSD]
                         + [(409600, 2, 3, 1e4)])
def test_kf_fuse_unimodal_matches_float64(rows, K, sd, kappa):
    """R11 (mmf_kf_fuse_unimodal): information-form fusion (models._information_fusion, +1e-9 elementwise) in float64.
    Covariances SPD with condition number <= kappa; on a seventh of the rows modality 0 is 1e4 times more confident.
    Above kappa = 1e2 each row is held to 8 kappa 2^-24 for the condition number it was built with."""
    regime = _fuse_regime(rows)
    g = torch.Generator(device=DEV).manual_seed(rows + 10 * K + sd + int(kappa))
    mu = torch.randn(K, rows, sd, device=DEV, generator=g)
    P, cond = _spd(K, rows, sd, kappa, g)
    if K > 1:
        P[0, ::7] *= 1e-4
    mean, cov = profiled(lambda: fuse_raw(K, rows, sd, mu, P, None), [f"k_kf_fuse<{sd}>"])
    mean_ref = M._information_fusion(mu.double(), P.double())
    cov_ref = torch.inverse(torch.inverse(P.double() + 1e-9).sum(0) + 1e-9)
    unit = cond.amax(0) * 2.0 ** -24  # a row's condition number times the fp32 unit roundoff
    bar = RTOL_R11 if kappa <= 1e2 else torch.clamp(KAPPA_FACTOR * unit, min=RTOL_R11)
    report, where = {}, _labels(("row", rows))
    report["/ (kappa 2^-24)"] = max(row_excess(mean, mean_ref, unit)[0],
                                    row_excess(cov.reshape(rows, -1), cov_ref.reshape(rows, -1), unit)[0])
    assert_rows(mean, mean_ref, bar, "mean", report, "mean", where)
    assert_rows(cov.reshape(rows, -1), cov_ref.reshape(rows, -1), bar, "cov", report, "cov", where)
    print(f"[K={K} sd={sd} rows={rows} kappa<={kappa:g}] {regime}; worst relative errors "
          + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("rows", FUSE_ROWS)
@pytest.mark.parametrize("K,sd", FUSE_KSD)
def test_kf_fuse_measurements_matches_float64(K, sd, rows):
    """R12 (mmf_kf_fuse_measurements) on the inputs of test_kf_fuse_measurements_matches_the_reference_expressions:
    crossmodal z and the Cholesky factor of models._measurement_level in float64; unimodal (K = 1: z_0 and L_0 L_0^T;
    K > 1: the reference's elementwise reciprocals, whose sum holds K 1e9 above the diagonal, inverted in float64)."""
    regime = _fuse_regime(rows)
    g = torch.Generator(device=DEV).manual_seed(71 + K + sd + rows)
    z = torch.randn(K, rows, sd, device=DEV, generator=g)
    tril = torch.tril(torch.randn(K, rows, sd, sd, device=DEV, generator=g)) * 0.3
    tril.diagonal(dim1=-2, dim2=-1).abs_().add_(0.2)
    w = torch.rand(K, rows, sd, device=DEV, generator=g) + 0.05
    where, report = _labels(("row", rows)), {}
    got_z, got_l = profiled(lambda: fuse_measurements_raw(K, rows, sd, z, tril, w), [f"k_kf_fuse_measurements<{sd}>"])
    ref_z, ref_cov = M._measurement_level(z.double(), tril.double(), w.double())
    assert_rows(got_z, ref_z, RTOL_R12_Z, "crossmodal z", report, "cross z", where)
    # a Cholesky factor in fp32 is good to about cond(C) 2^-24: each row is held to 8 times that, or RTOL_R12_Z
    unit = torch.linalg.cond(ref_cov) * 2.0 ** -24
    ref_l = torch.linalg.cholesky(ref_cov).reshape(rows, -1)
    report["cross factor / (cond 2^-24)"] = row_excess(got_l.reshape(rows, -1), ref_l, unit)[0]
    assert_rows(got_l.reshape(rows, -1), ref_l, torch.clamp(KAPPA_FACTOR * unit, min=RTOL_R12_FACTOR),
                "crossmodal factor", report, "cross factor", where)
    got_z, got_c = profiled(lambda: fuse_measurements_raw(K, rows, sd, z, tril, None), [f"k_kf_fuse_measurements<{sd}>"])
    t64 = tril.double()
    if K == 1:
        ref_z, ref_c = z[0].double(), t64[0] @ t64[0].mT
    else:
        prec = 1.0 / (tril + 1e-9)
        wd = torch.diagonal(prec, dim1=-2, dim2=-1).double()
        ref_z = (wd / (wd.sum(0) + 1e-9) * z.double()).sum(0)
        ref_c = torch.inverse(prec.double().sum(0) + 1e-9)
    assert_rows(got_z, ref_z, RTOL_R12_Z, "unimodal z", report, "uni z", where)
    assert_rows(got_c.reshape(rows, -1), ref_c.reshape(rows, -1), RTOL_R12_COV if K == 1 or sd < 4 else RTOL_R12_QUIRK,
                "unimodal covariance", report, "uni cov", where)
    print(f"[K={K} sd={sd} rows={rows}] {regime}; worst relative errors "
          + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- e. k_dyn_rollout, eval and tape, past 32 SMs trajectories -------------------------------------------------------
def rollout_raw(plan, x0, T, controls, rowbias, tape):
    N, sd = x0.shape
    chain, rows = plan.structs[0].dynamics, plan.structs[0].dynamics_rows
    states = _nan(T, N, sd)
    act = _nan(ops.dyn_depth(chain) + 1, U // 4, T * N, 4) if tape else None
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_dyn_rollout_fwd, C.byref(chain), C.byref(rows), T, N, _lib.ptr(x0), _lib.ptr(controls),
                         _lib.ptr(rowbias), _lib.ptr(states), _lib.ptr(act), _lib.stream_of(x0)))
    return states, act


@pytest.mark.gpu
@pytest.mark.parametrize("sd", [2, 3, 1, 4], ids=["push", "door", "sd1", "sd4"])
@pytest.mark.parametrize("path", ["rowbias", "controls"])
@pytest.mark.parametrize("T", [15, 100])
def test_dyn_rollout_matches_float64_teacher_forced(sd, path, T):
    """mmf_dyn_rollout_fwd at 4 rounds of 148 x 32 trajectories (the last one of 5), from given rows or from the controls
    (rows = NULL: the kernel's own control rows, the forward_loop path): every state from the float64 chain at the
    kernel's previous state; at T = 15 also the tape, every plane against the float64 input of its layer, and the eval
    states bit for bit against the tape forward's."""
    N = DYN_N
    plan = _ekf_plan(1, sd, seed=50 + sd)
    regime = dyn_regime(N, _plan_nf(plan), *_device())
    _assert_loops(regime)
    spec = plan.dyns[0]
    g = torch.Generator(device=DEV).manual_seed(N + T + sd)
    x0 = torch.randn(N, sd, device=DEV, generator=g)
    u = torch.randn(T, N, 7, device=DEV, generator=g)
    rows64 = torch.cat([control_rows64(spec, u.reshape(T * N, 7)[a:a + CHUNK]) for a in range(0, T * N, CHUNK)])
    rowbias = rows64.float().reshape(T, N, U).contiguous() if path == "rowbias" else None
    controls = u if path == "controls" else None
    states, _ = profiled(lambda: rollout_raw(plan, x0, T, controls, rowbias, tape=False), [f"k_dyn_rollout<{sd},false>"])
    act = None
    if T == 15:
        s_t, act = profiled(lambda: rollout_raw(plan, x0, T, controls, rowbias, tape=True), [f"k_dyn_rollout<{sd},true>"])
        assert torch.equal(states, s_t), "eval and tape rollout differ"
        act = ops.rows_view(act)  # (L+1, T N, 64)
    rb = rows64 if rowbias is None else rowbias.reshape(T * N, U).double()
    x_in = torch.cat([x0[None], states[:-1]]).reshape(T * N, sd)
    got, report, where = states.reshape(T * N, sd), {}, _labels(("t", T), ("n", N))
    for a in range(0, T * N, CHUNK):
        b = min(T * N, a + CHUNK)
        planes = [] if act is not None else None
        ref = dynamics64(spec, x_in[a:b], rb[a:b], planes=planes)
        at = lambda row: where(a + row)  # noqa: E731
        assert_rows(got[a:b], ref, RTOL_MEAN, "states", report, "states", at)
        for l, plane in enumerate(planes or []):
            assert_rows(act[l, a:b], plane, RTOL_PLANES, f"tape plane {l}", report, "planes", at)
    print(f"[sd={sd} {path} T={T}] N={N} {regime}; worst relative errors "
          + " ".join(f"{c} {v:.2e}" for c, v in report.items()))
