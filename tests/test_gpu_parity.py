"""Parity of the CUDA path (called through the C ABI) against the oracle, on identical inputs and
identical random draws.  Bar (BASELINE.json north_star): resampling indices BIT-EXACT; states,
covariances and log-likelihoods within 1e-4 relative in fp32 (see util.assert_close)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import crossmodal_port as port  # noqa: E402
from oracle import pinned  # noqa: E402
from oracle.golden_cases import run_all  # noqa: E402
from oracle.noise import RecordedNoise  # noqa: E402

from multimodalfilter_b200 import _lib, fused, ops  # noqa: E402
from multimodalfilter_b200.crossmodal import models as M  # noqa: E402
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories  # noqa: E402

from util import ReplayNoise, assert_close, draw_noise  # noqa: E402

DEV = "cuda:0"
RTOL = 1e-4


def _product(name):
    for task in M.MODEL_TYPES.values():
        if name in task:
            return task[name]
    return getattr(M, name)


def test_device_is_sm100_and_library_loads():
    lib = _lib.load()
    _lib.check(lib.mmf_device_check())
    assert torch.cuda.get_device_capability(0)[0] == 10


# ---- R2 ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,M,sd", [(5, 30, 2), (3, 300, 3), (1, 1, 2), (4096, 100, 2)])
def test_pf_init(N, M, sd):
    g = torch.Generator().manual_seed(N + M)
    mean = torch.randn(N, sd, generator=g)
    A = torch.randn(N, sd, sd, generator=g)
    cov = A @ A.transpose(-1, -2) + 0.1 * torch.eye(sd)
    eps = torch.randn(M, N, sd, generator=g)
    states, logw = ops.pf_init(mean.to(DEV), cov.to(DEV), eps.to(DEV))
    ref = (mean[None] + (torch.linalg.cholesky(cov)[None] @ eps[..., None]).squeeze(-1)).transpose(0, 1)
    assert_close(states.cpu(), ref, RTOL, msg="particle_states")
    assert torch.equal(logw.cpu(), torch.full((N, M), -math.log(M)))


# ---- R5 standalone -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,M,K,weighted", [(4, 7, 2, True), (3, 1000, 2, False), (2, 5, 3, True), (1, 1, 1, False)])
def test_fuse_loglik(N, M, K, weighted):
    g = torch.Generator().manual_seed(7)
    ll = torch.randn(N, M, K, generator=g) * 5
    w = torch.randn(N, K, generator=g) if weighted else None
    if weighted and K > 1:
        w[0, 0] = -float("inf")  # quirk Q3 blackout weight
    out = ops.fuse_loglik(ll.to(DEV), None if w is None else w.to(DEV))
    ref = torch.logsumexp(ll if w is None else w[:, None, :] + ll, dim=2)
    assert_close(out.cpu(), ref, RTOL, msg="fused log-likelihood")


# ---- R7 standalone: bit-exact indices ------------------------------------------------------------------
RESAMPLE_CASES = [(8, 30, 30), (4, 300, 300), (6, 1000, 1000), (3, 257, 64), (2, 1, 5), (5, 2, 9), (2, 4096, 4096), (1, 10000, 777),
                  (2, 70000, 5000), (1, 300000, 1000)]  # M > 2048: the multi-pass path of resample_big.cu (config C5); MMF_RESAMPLE_BIG=0
#                                         sends them through the CTA-per-trajectory kernels instead (tools/gpu_validate.sh runs both)


@pytest.mark.parametrize("mode", ["multinomial", "multinomial_fast", "systematic", "systematic_fast"])
@pytest.mark.parametrize("N,M,S", RESAMPLE_CASES)
def test_resample_indices_bit_exact(mode, N, M, S):
    g = torch.Generator().manual_seed(1000 * N + M)
    logits = torch.randn(N, M, generator=g) * 4
    logits = logits - torch.logsumexp(logits, dim=1, keepdim=True)
    if M > 3:
        logits[0, 1] = -float("inf")      # a dead particle
        logits[-1, : M // 2] = -200.0     # underflowing mass
    u = torch.rand(N, generator=g, dtype=torch.float64) if mode.startswith("systematic") else \
        torch.rand(N, S, generator=g, dtype=torch.float64)
    idx = ops.resample_indices(logits.to(DEV), u.to(DEV), mode=ops.RESAMPLE_MODES[mode], M_out=S).cpu().numpy()
    ref = pinned.resample(logits.numpy(), u.numpy(), mode, num_samples=S)
    assert idx.shape == ref.shape == (N, S)
    assert np.array_equal(idx, ref), f"{(idx != ref).sum()} / {idx.size} indices differ"
    assert idx.min() >= 0 and idx.max() < M
    if M > 3:
        assert not (idx[0] == 1).any()  # the dead particle is never drawn


def test_resample_degenerate_distributions():
    M = 64
    logits = torch.full((3, M), -float("inf"))
    logits[0, 17] = 0.0                      # one-hot
    logits[1] = -math.log(M)                 # exactly uniform
    logits[2, [3, 60]] = math.log(0.5)       # two atoms
    u = torch.rand(3, M, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    for mode in ("multinomial", "multinomial_fast"):
        idx = ops.resample_indices(logits.to(DEV), u.to(DEV), mode=ops.RESAMPLE_MODES[mode]).cpu()
        assert (idx[0] == 17).all()
        assert set(idx[2].tolist()) <= {3, 60}
        assert np.array_equal(idx.numpy(), pinned.resample(logits.numpy(), u.numpy(), mode))
    u0 = torch.tensor([0.25, 0.5, 0.999], dtype=torch.float64)
    idx = ops.resample_indices(logits.to(DEV), u0.to(DEV), mode=ops.RESAMPLE_SYSTEMATIC_STRICT).cpu()
    assert torch.equal(idx[1], torch.arange(M))  # uniform weights + systematic = identity


def test_pinned_arithmetic_differs_from_torch_only_at_cdf_ties():
    """The pinned CDF and torch.multinomial's CPU CDF agree except where a uniform falls within
    rounding distance of a CDF step (SURVEY.md section 7, hard part 1c)."""
    N, M = 64, 1000
    g = torch.Generator().manual_seed(11)
    logits = torch.randn(N, M, generator=g) * 3
    logits = logits - torch.logsumexp(logits, dim=1, keepdim=True)
    u = torch.rand(N, M, generator=g, dtype=torch.float64)
    idx = ops.resample_indices(logits.to(DEV), u.to(DEV)).cpu().numpy()
    probs = torch.softmax(logits, dim=-1)
    from torchfilter.filters import multinomial_inverse_cdf

    ref = multinomial_inverse_cdf(probs, u).numpy()
    diff = np.argwhere(idx != ref)
    assert len(diff) < 1e-3 * idx.size
    cdf = np.cumsum(probs.numpy().astype(np.float64), axis=1)
    for n, j in diff:
        lo, hi = sorted((idx[n, j], ref[n, j]))
        assert hi - lo == 1 and abs(cdf[n, lo] - u[n, j].item()) < 2e-6


# ---- R6 + R7 fused kernel ----------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["none", "multinomial", "multinomial_fast", "systematic"])
@pytest.mark.parametrize("N,M,sd,M_out,alpha,estimation", [
    (6, 30, 2, 30, 1.0, "weighted_average"),
    (4, 300, 3, 300, 1.0, "weighted_average"),
    (3, 1000, 2, 1000, 1.0, "argmax"),
    (5, 30, 2, 300, 1.0, "weighted_average"),   # eval after train: particle count grows (quirk Q8)
    (4, 100, 3, 100, 0.5, "weighted_average"),  # soft resampling
    (2, 1, 2, 1, 1.0, "weighted_average"),
    (2, 100000, 2, 100000, 1.0, "weighted_average"),  # global-workspace path
])
def test_normalize_estimate_resample(mode, N, M, sd, M_out, alpha, estimation):
    if mode == "none" and (M_out != M or alpha != 1.0):
        pytest.skip("no resampling: count / alpha irrelevant")
    g = torch.Generator().manual_seed(N * M + sd)
    states = torch.randn(N, M, sd, generator=g)
    logw_unnorm = torch.randn(N, M, generator=g) * 3 - 5
    code = ops.RESAMPLE_NONE if mode == "none" else ops.RESAMPLE_MODES[mode]
    u = None
    if mode != "none":
        u = torch.rand(N, generator=g, dtype=torch.float64) if mode.startswith("systematic") else \
            torch.rand(N, M_out, generator=g, dtype=torch.float64)
    out = ops.pf_normalize_resample(states.to(DEV), logw_unnorm.to(DEV), estimation=ops.ESTIMATION[estimation],
                                    mode=code, alpha=alpha, M_out=M_out, uniforms=None if u is None else u.to(DEV),
                                    want_debug=True)
    logw = logw_unnorm - torch.logsumexp(logw_unnorm, dim=1, keepdim=True)
    assert_close(out["logw_norm"].cpu(), logw, RTOL, msg="normalised log-weights")
    if estimation == "weighted_average":
        est = torch.sum(torch.exp(logw)[:, :, None] * states, dim=1)
        assert_close(out["estimate"].cpu(), est, RTOL, msg="estimate")
    else:
        best = torch.argmax(logw, dim=1)
        assert torch.equal(out["estimate"].cpu(), states[torch.arange(N), best])
    if mode == "none":
        assert_close(out["logw"].cpu(), logw, RTOL, msg="log-weights")
        return
    if alpha < 1.0:
        uniform = torch.full((N, M), -math.log(M))
        logits = torch.logsumexp(torch.stack([logw + math.log(alpha), uniform + math.log(1 - alpha)]), dim=0)
        assert_close(out["logits"].cpu(), logits, RTOL, msg="soft-resampling logits")
    # indices: bit-exact against the pinned arithmetic applied to the kernel's own logits
    ref_idx = pinned.resample(out["logits"].cpu().numpy(), u.numpy(), mode, num_samples=M_out)
    idx = out["idx"].cpu().numpy()
    assert np.array_equal(idx, ref_idx), f"{(idx != ref_idx).sum()} / {idx.size} indices differ"
    gathered = torch.gather(states, 1, torch.from_numpy(idx)[:, :, None].expand(N, M_out, sd))
    assert torch.equal(out["states"].cpu(), gathered)  # a gather moves bits, it must be exact
    if alpha < 1.0:
        new_logw = torch.gather(out["logw_norm"].cpu() - out["logits"].cpu(), 1, torch.from_numpy(idx))
        assert_close(out["logw"].cpu(), new_logw, 1e-5, msg="soft-resampled log-weights")
    else:
        assert torch.equal(out["logw"].cpu(), torch.full((N, M_out), -math.log(M)))


# ---- R3 + R4 + R5 per-particle chain -------------------------------------------------------------------
@pytest.mark.parametrize("name,sd,flags", [
    ("PushCrossmodalParticleFilter", 2, [True, True]),
    ("PushCrossmodalParticleFilter", 2, [False, True]),
    ("PushCrossmodalParticleFilterSeq5", 2, [True, True]),
    ("DoorCrossmodalParticleFilter", 3, [True, True]),
    ("PushUnimodalParticleFilter", 2, [True, True]),
    ("DoorUnimodalParticleFilter", 3, [True, False]),
    ("PushParticleFilter", 2, None),
])
@pytest.mark.parametrize("N,Mp", [(5, 30), (3, 300), (2, 1000)])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_predict_measure_matches_oracle_modules(name, sd, flags, N, Mp, precision):
    oracle_f = fill_parameters(getattr(port, name)(), seed=21).eval()
    prod_f = fill_parameters(_product(name)(), seed=21).to(DEV).eval()
    if flags is not None:
        oracle_f.measurement_model.enabled_models = list(flags)
        prod_f.measurement_model.enabled_models = list(flags)
    g = torch.Generator().manual_seed(5 * N + Mp)
    states = torch.randn(N, Mp, sd, generator=g)
    logw = torch.randn(N, Mp, generator=g) - 3
    eps = torch.randn(N * Mp, sd, generator=g)
    _, obs, controls = synthetic_trajectories(1, N, sd, seed=31, blackout_fraction=0.4 if "Seq5" in name else 0.0)
    obs0, u0 = {k: v[0] for k, v in obs.items()}, controls[0]

    with torch.no_grad():
        pred, trils = oracle_f.dynamics_model(initial_states=states.reshape(-1, sd),
                                              controls=u0.repeat_interleave(Mp, dim=0))
        moved = (pred + (trils @ eps[..., None]).squeeze(-1)).view(N, Mp, sd)
        ll = oracle_f.measurement_model(states=moved, observations=obs0)
        ref_logw = logw + ll

    plan = fused.PFPlan.build(prod_f)
    assert plan is not None
    plan.refresh(torch.device(DEV))
    obs_d = {k: v.to(DEV) for k, v in obs0.items()}
    with torch.no_grad():
        feats = plan.head_features(obs_d)
        modw = plan.modality_log_weights(obs_d)
    rowbias = ops.pf_traj_rows(plan.struct, plan.K, u0.to(DEV), feats)
    moved_k, logw_k, ll_k = ops.pf_predict_measure(plan.struct, states.to(DEV), eps.to(DEV), rowbias, logw.to(DEV),
                                                   modw, plan.enabled_mask(), precision=ops.PRECISIONS[precision],
                                                   want_ll=True)
    # fp32 (CUDA cores) and bf16x3 (tcgen05, split operands) are parity grade; single-pass bf16 is the
    # opt-in fast mode and is only held to bf16 accuracy (8 mantissa bits through ~10 layers)
    RTOL = 1e-4 if precision != "bf16" else 3e-2
    assert_close(moved_k.cpu(), moved, RTOL, msg="moved particle states")
    assert_close(logw_k.cpu(), ref_logw, RTOL, msg="un-normalised log-weights")
    # per-head log-likelihoods against the oracle's individual heads
    mm = oracle_f.measurement_model
    heads = list(mm.measurement_models) if hasattr(mm, "measurement_models") else [mm]
    for k, head in enumerate(heads):
        if flags is not None and not flags[k]:
            assert torch.isnan(ll_k[k]).all()  # never written
            continue
        with torch.no_grad():
            assert_close(ll_k[k].cpu(), head(states=moved, observations=obs0), RTOL, msg=f"head {k} log-likelihood")


# ---- golden fixture (generated by the reference's own code) ---------------------------------------
@pytest.mark.parametrize("group", ["dyn/", "head/", "fuse/", "vsensor/", "kf/"])
def test_product_matches_reference_fixture(golden, group):
    got = run_all(_product, device=DEV, include_rng_cases=False, only=[group])
    keys = [k for k in golden if k.startswith(group)]
    assert sorted(got) == sorted(keys)
    for k in keys:
        assert_close(got[k], golden[k], RTOL, msg=k)


# ---- whole recursion, PF ---------------------------------------------------------------------------------
def _run_pair(name, sd, N, Mp, T, train, mode="multinomial", seed=3):
    init, eps, us = draw_noise(T, N, Mp, sd, seed=seed, systematic=mode.startswith("systematic"))
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=seed + 1)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd)

    o = fill_parameters(getattr(port, name)(), seed=22)
    o.train(train)
    o.num_particles = Mp
    o.noise = RecordedNoise(init_eps=init, process_eps=eps, uniforms=us, mode=mode, arithmetic="pinned")
    with torch.no_grad():
        o.initialize_beliefs(mean=states[0], covariance=cov)
        ref = o.forward_loop(observations={k: v[1:] for k, v in obs.items()}, controls=controls[1:])

    p = fill_parameters(_product(name)(), seed=22).to(DEV)
    p.train(train)
    p.num_particles = Mp
    p.resample_mode = mode
    p.noise = ReplayNoise(init_eps=init, process_eps=eps, uniforms=us)
    with torch.no_grad():
        p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov.to(DEV).contiguous())
        got = p.forward_loop(observations={k: v[1:].to(DEV) for k, v in obs.items()}, controls=controls[1:].to(DEV))
    return o, ref, p, got


@pytest.mark.parametrize("name,sd", [("PushCrossmodalParticleFilter", 2), ("DoorCrossmodalParticleFilter", 3),
                                     ("PushUnimodalParticleFilter", 2)])
def test_forward_loop_train_mode_no_resampling(name, sd):
    o, ref, p, got = _run_pair(name, sd, N=6, Mp=30, T=8, train=True)
    assert_close(got.cpu(), ref, RTOL, msg="estimates")
    assert_close(p.particle_states.cpu(), o.particle_states, RTOL, msg="particle states")
    assert_close(p.particle_log_weights.cpu(), o.particle_log_weights, RTOL, msg="particle log-weights")


@pytest.mark.parametrize("mode", ["multinomial", "multinomial_fast", "systematic"])
@pytest.mark.parametrize("name,sd,Mp", [("PushCrossmodalParticleFilter", 2, 30), ("DoorCrossmodalParticleFilter", 3, 300)])
def test_filter_steps_eval_mode_with_resampling(name, sd, Mp, mode):
    """BASELINE config C1 in miniature: crossmodal PF eval, resampling every step, identical draws.

    Both filters start every step from the SAME particle set (the oracle's), so float differences
    cannot compound through resampling.  Estimates must agree to 1e-4; resampling indices must be
    identical, except where a uniform sits within rounding distance of a CDF step -- there the
    1e-6-level difference between the CPU oracle's and the kernel's *logits* may pick the
    neighbouring particle; every such case is checked to be exactly that (and they are rare)."""
    N, T = 8, 10
    init, eps, us = draw_noise(T, N, Mp, sd, seed=3, systematic=mode.startswith("systematic"))
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=4)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd)
    o = fill_parameters(getattr(port, name)(), seed=22).eval()
    o.num_particles = Mp
    o.noise = RecordedNoise(init_eps=init, process_eps=eps, uniforms=us, mode=mode, arithmetic="pinned")
    p = fill_parameters(_product(name)(), seed=22).to(DEV).eval()
    p.num_particles = Mp
    p.resample_mode = mode
    p.noise = ReplayNoise(init_eps=init, process_eps=eps, uniforms=us)
    p.debug = {}
    draws = flips = 0
    with torch.no_grad():
        o.initialize_beliefs(mean=states[0], covariance=cov)
        p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov.to(DEV).contiguous())
        assert_close(p.particle_states.cpu(), o.particle_states, RTOL, msg="initial particles")
        for t in range(T):
            p.particle_states = o.particle_states.to(DEV).contiguous()
            p.particle_log_weights = o.particle_log_weights.to(DEV).contiguous()
            obs_t = {k: v[1 + t] for k, v in obs.items()}
            est_o = o(observations=obs_t, controls=controls[1 + t])
            est_p = p(observations={k: v.to(DEV) for k, v in obs_t.items()}, controls=controls[1 + t].to(DEV))
            assert_close(est_p.cpu(), est_o, RTOL, msg=f"estimate at step {t}")
            idx_o, idx_p = o.noise.indices[-1], p.debug["idx"].cpu()
            same = (idx_o == idx_p).all(dim=1)
            draws += idx_o.numel()
            if not same.all():
                # prove each differing draw is a CDF tie on the kernel's own logits
                u = us[t].numpy()
                _, cdf = pinned.resample(p.debug["logits"].cpu().numpy(), u, mode, num_samples=Mp, return_cdf=True)
                for n, j in np.argwhere((idx_o != idx_p).numpy()):
                    flips += 1
                    lo, hi = sorted((int(idx_o[n, j]), int(idx_p[n, j])))
                    assert hi - lo == 1, "indices differ by more than one slot"
                    uj = (u[n] + j) / Mp if mode.startswith("systematic") else u[n, j]
                    assert abs(cdf[n, lo] / cdf[n, -1] - uj) < 5e-6, "index differs away from a CDF tie"
            assert_close(p.particle_states.cpu()[same], o.particle_states[same], RTOL, msg=f"resampled states, step {t}")
            assert torch.equal(p.particle_log_weights.cpu(), o.particle_log_weights)
    assert flips <= max(2, draws // 5000), f"{flips} tie flips in {draws} draws"


def test_single_step_forward_equals_forward_loop():
    name, sd, N, Mp, T = "PushCrossmodalParticleFilter", 2, 4, 30, 4
    init, eps, us = draw_noise(T, N, Mp, sd, seed=9)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=10)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    outs = []
    for use_loop in (True, False):
        p = fill_parameters(_product(name)(), seed=23).to(DEV).eval()
        p.num_particles = Mp
        p.noise = ReplayNoise(init_eps=init, process_eps=eps, uniforms=us)
        with torch.no_grad():
            p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
            o_d = {k: v[1:].to(DEV) for k, v in obs.items()}
            if use_loop:
                outs.append(p.forward_loop(observations=o_d, controls=controls[1:].to(DEV)))
            else:
                outs.append(torch.stack([p(observations={k: v[t] for k, v in o_d.items()},
                                           controls=controls[1 + t].to(DEV)) for t in range(T)]))
    # the hoisted encoders run on T*N rows, the per-step ones on N rows: library GEMMs may block differently
    assert_close(outs[0].cpu(), outs[1].cpu(), 1e-5, msg="hoisted vs per-step")


# ---- whole recursion, EKF (BASELINE config C2 in miniature) -------------------------------------------
@pytest.mark.parametrize("name,sd", [("DoorCrossmodalKalmanFilter", 3), ("PushCrossmodalKalmanFilter", 2),
                                     ("DoorUnimodalKalmanFilter", 3), ("DoorKalmanFilter", 3)])
def test_ekf_forward_loop_matches_oracle(name, sd):
    T, N = 20, 16
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=12)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd)
    o = fill_parameters(getattr(port, name)(), seed=24).eval()
    with torch.no_grad():
        o.initialize_beliefs(mean=states[0], covariance=cov)
        ref = o.forward_loop(observations={k: v[1:] for k, v in obs.items()}, controls=controls[1:])
    p = fill_parameters(_product(name)(), seed=24).to(DEV).eval()
    with torch.no_grad():
        p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov.to(DEV).contiguous())
        got = p.forward_loop(observations={k: v[1:].to(DEV) for k, v in obs.items()}, controls=controls[1:].to(DEV))
    assert_close(got.cpu(), ref, RTOL, msg="EKF estimates")
    ocov = getattr(o, "weighted_covariances", None)
    pcov = getattr(p, "weighted_covariances", None)
    if ocov is not None and pcov is not None:
        assert_close(pcov.cpu(), ocov, RTOL, msg="fused covariance")
    of = list(o.filter_models) if hasattr(o, "filter_models") else [o]
    pf = list(p.filter_models) if hasattr(p, "filter_models") else [p]
    for a, b in zip(of, pf):
        assert_close(b.belief_mean.cpu(), a.belief_mean, RTOL, msg="unimodal belief mean")
        assert_close(b.belief_covariance.cpu(), a.belief_covariance, RTOL, msg="unimodal belief covariance")


def test_dynamics_jacobian_kernel_matches_autograd():
    dyn_o = fill_parameters(port.DoorDynamicsModel(), seed=25)
    dyn_p = fill_parameters(M.DoorDynamicsModel(), seed=25).to(DEV)
    x, u = torch.randn(33, 3), torch.randn(33, 7)
    ref = dyn_o.jacobian(initial_states=x, controls=u).detach()
    with torch.no_grad():
        got = dyn_p.jacobian(initial_states=x.to(DEV), controls=u.to(DEV))
    assert_close(got.cpu(), ref, RTOL, msg="dynamics Jacobian")


# ---- size-independent properties at BASELINE sizes -----------------------------------------------------
def test_full_size_step_properties_and_shard_invariance():
    """Config C3 shape (N=4096, M=1000, sd=2), one step: normalised weights, sortedness of
    systematic indices, and trajectory-sharded == unsharded bit-for-bit (SURVEY.md section 8e)."""
    N, Mp, sd = 4096, 1000, 2
    p = fill_parameters(M.PushUnimodalParticleFilter(), seed=26).to(DEV).eval()
    plan = fused.PFPlan.build(p)
    plan.refresh(torch.device(DEV))
    g = torch.Generator(device=DEV).manual_seed(0)
    states = torch.randn(N, Mp, sd, device=DEV, generator=g)
    logw = torch.full((N, Mp), -math.log(Mp), device=DEV)
    eps = torch.randn(N * Mp, sd, device=DEV, generator=g)
    controls = torch.randn(N, 7, device=DEV, generator=g)
    feats = [torch.randn(N, 64, device=DEV, generator=g), torch.randn(N, 128, device=DEV, generator=g)]
    u = torch.rand(N, device=DEV, dtype=torch.float64, generator=g)

    def step(lo, hi):
        rb = ops.pf_traj_rows(plan.struct, 2, controls[lo:hi], [f[lo:hi] for f in feats])
        moved, lw = ops.pf_predict_measure(plan.struct, states[lo:hi], eps[lo * Mp:hi * Mp], rb, logw[lo:hi], None, 3)
        out = ops.pf_normalize_resample(moved, lw, mode=ops.RESAMPLE_SYSTEMATIC_FAST, uniforms=u[lo:hi], want_debug=True)
        return moved, lw, out

    moved, lw, out = step(0, N)
    assert torch.isfinite(moved).all() and torch.isfinite(lw).all()
    total = torch.exp(out["logw_norm"].double()).sum(dim=1)
    assert (total - 1).abs().max() < 1e-4
    idx = out["idx"]
    assert (idx[:, 1:] >= idx[:, :-1]).all() and idx.min() >= 0 and idx.max() < Mp
    counts = torch.zeros(N, Mp, device=DEV).scatter_add_(1, idx, torch.ones_like(idx, dtype=torch.float32))
    expected = torch.exp(out["logw_norm"]) * Mp
    assert (counts - expected).abs().max() <= 1.0 + 1e-3  # systematic resampling: |count - M w| <= 1
    half = N // 2
    a, b = step(0, half), step(half, N)
    assert torch.equal(torch.cat([a[0], b[0]]), moved)
    assert torch.equal(torch.cat([a[1], b[1]]), lw)
    for key in ("states", "estimate", "idx", "logw_norm"):
        assert torch.equal(torch.cat([a[2][key], b[2][key]]), out[key]), key


# ---- training path: gradients through the recursion (BPTT, BASELINE config C4 in miniature) ---------
@pytest.mark.parametrize("freeze_dynamics", [False, True])
def test_bptt_gradients_match_oracle(freeze_dynamics):
    """freeze_dynamics=True is the reference's actual end-to-end setting and takes the fused training step
    (mmf_pf_heads_forward_train / mmf_pf_heads_backward); False exercises the generic autograd path.

    PushCrossmodalParticleFilter.train(): no resampling, MSE on the estimates, backward through all steps.
    Gradients of the measurement / weight-model parameters (the ones the reference's curricula train; the
    dynamics is frozen there, ref: scripts/push_task/train_push.py:154) and of the dynamics parameters
    must match the CPU oracle's autograd."""
    # The fused path evaluates the heads in split-bf16 (1e-5 relative): over many steps a pre-activation that
    # sits within that distance of zero can take the other side of its ReLU than in the fp32 oracle, which changes
    # that particle's gradient below the flipped unit by O(1).  T = 3 keeps the comparison free of such flips
    # (seen from T = 4 on with these seeds); the kernel itself is checked flip-free, layer by layer, in
    # test_heads_backward_kernel_matches_autograd.
    name, sd, N, Mp, T = "PushCrossmodalParticleFilter", 2, 6, 30, (3 if freeze_dynamics else 5)
    init, eps, _ = draw_noise(T, N, Mp, sd, seed=13)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=14)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd)
    grads = []
    for side in ("oracle", "product"):
        if side == "oracle":
            f = fill_parameters(getattr(port, name)(), seed=27)
            f.noise = RecordedNoise(init_eps=init, process_eps=eps)
            dev = "cpu"
        else:
            f = fill_parameters(_product(name)(), seed=27).to(DEV)
            f.noise = ReplayNoise(init_eps=init, process_eps=eps)
            dev = DEV
        f.train()
        f.num_particles = Mp
        if freeze_dynamics:
            for prm in f.dynamics_model.parameters():
                prm.requires_grad_(False)
        if side == "product":
            from multimodalfilter_b200 import ops as _ops

            _ops.PROFILE.reset(enabled=False)
        f.initialize_beliefs(mean=states[0].to(dev), covariance=cov.to(dev).contiguous())
        est = f.forward_loop(observations={k: v[1:].to(dev) for k, v in obs.items()}, controls=controls[1:].to(dev))
        loss = torch.mean((est - states[1:].to(dev)) ** 2)
        loss.backward()
        grads.append((loss.item(), {k: p.grad.detach().cpu() for k, p in f.named_parameters() if p.grad is not None}))
    (lo, go), (lp, gp) = grads
    assert abs(lo - lp) <= 1e-4 * abs(lo)
    assert set(go) == set(gp) and len(go) > 50
    if freeze_dynamics:  # the fused kernels must actually have run (T steps forward, T steps backward)
        assert _ops.PROFILE.launches >= 3 * T and not any(k.startswith("dynamics_model") for k in gp)
    # gradients span many orders of magnitude across the tree (the image-encoder convolutions see ~1e-7):
    # compare each tensor relative to its own scale, with an absolute floor tied to the largest gradient
    floor = 1e-5 * max(float(g.abs().max()) for g in go.values())
    for k in go:
        assert_close(gp[k], go[k], 2e-3, atol=floor, msg=f"grad {k}")


def test_heads_backward_kernel_matches_autograd():
    """mmf_pf_heads_forward_train / mmf_pf_heads_backward against torch autograd on the same chain, per layer:
    saved activations, per-head log-likelihoods, and the delta of every layer's pre-activation."""
    import torch.nn.functional as F

    for name, sd in (("PushCrossmodalParticleFilter", 2), ("DoorCrossmodalParticleFilter", 3)):
        f = fill_parameters(_product(name)(), seed=27).to(DEV)
        plan = fused.PFPlan.build(f)
        plan.refresh(torch.device(DEV), backward=True)
        N, Mp = 7, 50  # 350 rows: two full tiles and a ragged one
        g = torch.Generator(device=DEV).manual_seed(1)
        states = torch.randn(N, Mp, sd, device=DEV, generator=g)
        eps = torch.randn(N * Mp, sd, device=DEV, generator=g)
        rows = torch.randn(1 + plan.K, N, 64, device=DEV, generator=g)
        moved, ll, act = ops.pf_heads_forward_train(plan.struct, states, eps, rows, 3)
        d_ll = torch.randn(plan.K, N, Mp, device=DEV, generator=g)
        delta = ops.pf_heads_backward(plan.struct, N, Mp, act, d_ll, 3)
        dW, db, g_in, g_out = ops.pf_heads_weight_grads(act, delta, moved.reshape(-1, sd), d_ll.reshape(plan.K, -1))
        act_r, delta_r = ops.rows_view(act), ops.rows_view(delta)  # chunk-major planes -> (K, L+1, P, 64)
        x = moved.reshape(-1, sd)
        for k, spec in enumerate(plan.heads):
            (in_lin, pre), (mid, post, out) = spec.state, spec.shared
            zs, acts = [], []

            def lin(w, b, a):
                z = F.linear(a, w, b)
                z.retain_grad()
                zs.append(z)
                return z

            a = torch.relu(lin(in_lin.weight, in_lin.bias, x))
            acts.append(a)
            for r in pre:
                t = torch.relu(lin(r.block1.weight, r.block1.bias, a))
                acts.append(t)
                a = torch.relu(lin(r.block2.weight, r.block2.bias, t) + a)
                acts.append(a)
            z = F.linear(a, mid.weight[:, spec.feat_dim:]) + rows[1 + k].repeat_interleave(Mp, dim=0)
            z.retain_grad()
            zs.append(z)
            a = torch.relu(z)
            acts.append(a)
            for r in post:
                t = torch.relu(lin(r.block1.weight, r.block1.bias, a))
                acts.append(t)
                a = torch.relu(lin(r.block2.weight, r.block2.bias, t) + a)
                acts.append(a)
            llk = F.linear(a, out.weight, out.bias)[:, 0]
            assert_close(ll[k].reshape(-1).cpu(), llk.detach().cpu(), RTOL, msg=f"{name} head {k} log-likelihood")
            (llk * d_ll[k].reshape(-1)).sum().backward()
            L = len(zs) - 1
            for i, a_ref in enumerate(acts):
                assert_close(act_r[k, i].cpu(), a_ref.detach().cpu(), RTOL, msg=f"{name} head {k} activation {i}")
            for l in range(L):
                assert_close(delta_r[k, l].cpu(), zs[1 + l].grad.cpu(), 2e-4, msg=f"{name} head {k} delta {l}")
                # weight gradient of layer l: delta_l^T a_l (fp32 reduction in mmf_pf_heads_weight_grads)
                assert_close(dW[k, l].cpu(), (zs[1 + l].grad.t() @ acts[l].detach()).cpu(), 2e-4,
                             msg=f"{name} head {k} dW {l}")
            assert_close(delta_r[k, L].cpu(), zs[0].grad.cpu(), 2e-4, msg=f"{name} head {k} input-layer delta")
            # thin layers at both ends and the biases (mmf_pf_heads_weight_grads, second kernel)
            assert_close(g_in[k].cpu(), in_lin.weight.grad.cpu(), 2e-4, msg=f"{name} head {k} input-layer weight grad")
            assert_close(db[k, L].cpu(), in_lin.bias.grad.cpu(), 2e-4, msg=f"{name} head {k} input-layer bias grad")
            assert_close(g_out[k][None].cpu(), out.weight.grad.cpu(), 2e-4, msg=f"{name} head {k} output-layer weight grad")
            assert_close(db[k, 0].cpu(), zs[1].grad.sum(0).cpu(), 2e-4, msg=f"{name} head {k} bias grad of layer 0")


# ---- image encoder trunk (SURVEY.md 8(f)-1): tcgen05 implicit-GEMM convolutions vs torch fp32 ---------------
# A 32-channel activation map is [chunk of 8 channels 4][hi|lo][1280 positions][8 bf16]: a 64-position zero guard, then
# position 34 y + x (two zero pad columns per row), then zeros.  mmf_enc_trunk's scratch holds four such maps per CTA.
MAP32 = 4 * 2 * 1280 * 16  # 163,840 B


def _unmap(maps):
    """(m, MAP32) uint8 maps -> (m, 32, 32, 32) fp32 = hi + lo of every channel at every pixel"""
    t = maps.view(torch.bfloat16).reshape(-1, 4, 2, 1280, 8).float()
    v = (t[:, :, 0] + t[:, :, 1])[:, :, 64:64 + 1088].reshape(-1, 4, 32, 34, 8)[:, :, :, :32]
    return v.permute(0, 1, 4, 2, 3).reshape(-1, 32, 32, 32)


@pytest.mark.parametrize("n", [1, 37, 300])
def test_encoder_trunk_layers_match_torch(n):
    """Every layer of the fused trunk, read out of its own scratch: per CTA [x buf 0 | x buf 1 | t, later z | y].  CTA c
    runs images c, c + G, ...; the k-th of them has its stem output in x[k & 1], so after the launch the maps hold
    each CTA's last image (and, in the other x buffer, the previous one's stem output)."""
    import torch.nn.functional as F
    torch.manual_seed(n)
    img = (torch.rand(n, 32, 32, device=DEV) * 2 - 1).contiguous()
    img[0, :3] = 0.0
    c1 = torch.nn.Conv2d(1, 32, 5, padding=2).to(DEV)
    c2a, c2b = torch.nn.Conv2d(32, 32, 3, padding=1).to(DEV), torch.nn.Conv2d(32, 32, 3, padding=1).to(DEV)
    c3, c4 = torch.nn.Conv2d(32, 16, 3, padding=1).to(DEV), torch.nn.Conv2d(16, 8, 3, padding=1).to(DEV)
    tol = 5e-5  # activations are kept as bf16 hi + lo (2^-18 relative); accumulation is fp32
    with torch.no_grad():
        x_ref = F.relu(c1(img[:, None]))
        t_ref = F.relu(c2a(x_ref))
        y_ref = F.relu(c2b(t_ref) + x_ref)
        z_ref = F.relu(c3(y_ref))
        out_ref = c4(z_ref)
        w = ops.enc_pack_trunk([c1, c2a, c2b, c3, c4])
        scratch = ops.enc_trunk_scratch(DEV)
        out = ops.enc_trunk(img, w, scratch, 8)
        maps = scratch.cpu()
    assert maps.numel() % (4 * MAP32) == 0
    g_max = maps.numel() // (4 * MAP32)
    G = min(g_max, n)
    maps = maps.view(g_max, 4, MAP32)[:G]
    ctas = torch.arange(G)
    k_last = torch.tensor([len(range(c, n, G)) - 1 for c in range(G)])
    last = ctas + G * k_last
    x_last = _unmap(maps[ctas, k_last & 1])
    tz = _unmap(maps[:, 2])
    assert_close(x_last, x_ref[last].cpu(), tol, msg="layer 0: 5x5 stem + ReLU (x)")
    assert_close(tz[:, 16:], t_ref[last, 16:].cpu(), tol, msg="layer 1: block1 32->32 + ReLU (t, channels 16-31)")
    assert_close(_unmap(maps[:, 3]), y_ref[last].cpu(), tol, msg="layer 2: block2 32->32 + residual + ReLU (y)")
    assert_close(tz[:, :16], z_ref[last].cpu(), tol, msg="layer 3: 32->16 + ReLU (z)")
    # the previous image of a CTA left its stem output in the other x buffer (double-buffering parity)
    prev = k_last >= 1
    assert bool(prev.any()) == (n > G)
    if n > G:
        x_prev = _unmap(maps[ctas[prev], (k_last[prev] - 1) & 1])
        assert_close(x_prev, x_ref[last[prev] - G].cpu(), tol, msg="layer 0 of the previous image (other x buffer)")
    assert_close(out.cpu(), out_ref.cpu(), tol, msg="layer 4: 16->8 (NCHW output)")
    assert torch.equal(out, ops.enc_trunk(img, w, scratch, 8)), "fused trunk is not deterministic / scratch reuse"
    # the zero guards and the pad columns of every scratch map are still zero (the next layer's padding depends on it)
    planes = maps.view(G, 4, 8, 1280, 16)
    assert int(planes[..., :64, :].count_nonzero()) == 0 and int(planes[..., 64 + 1088:, :].count_nonzero()) == 0
    assert int(planes[..., 64:64 + 1088, :].reshape(G, 4, 8, 32, 34, 16)[..., 32:, :].count_nonzero()) == 0


@pytest.mark.parametrize("batch", [3, 16384 + 5])
def test_image_encoder_module_fused_trunk_matches_torch_path(batch):
    from multimodalfilter_b200.encoders import ImageEncoder
    filt = fill_parameters(M.PushCrossmodalParticleFilter(), seed=3).to(DEV).eval()
    enc = filt.measurement_model.measurement_models[0].observation_image_layers
    assert isinstance(enc, ImageEncoder) and enc._trunk() is not None
    g = torch.Generator(device=DEV).manual_seed(batch)
    x = torch.rand(batch, 1, 32, 32, device=DEV, generator=g) * 2 - 1
    x[1] = 0.0  # a blacked-out image
    with torch.no_grad():
        ops.PROFILE.reset(enabled=True)
        fused_out = enc(x)
        launched = ops.PROFILE.collect()["launches"]
        ops.PROFILE.reset(enabled=False)
        enc.fused_trunk = False
        try:
            torch_out = enc(x)
        finally:
            del enc.fused_trunk
    assert launched >= 1, "the fused trunk did not run"
    assert_close(fused_out.cpu(), torch_out.cpu(), 5e-5, msg="encoder features")
    # with autograd on the module is the plain torch Sequential (training path untouched)
    y = enc(x[:2])
    assert y.requires_grad


def test_forward_loop_streams_host_observations():
    """Pinned host observations are staged chunk by chunk behind the encoders; the result is that of device inputs."""
    name, sd, N, Mp, T = "PushCrossmodalParticleFilter", 2, 6, 30, 5
    init, eps, us = draw_noise(T, N, Mp, sd, seed=4)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=5)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    outs = []
    for host in (False, True):
        p = fill_parameters(_product(name)(), seed=23).to(DEV).eval()
        p.num_particles = Mp
        p.noise = ReplayNoise(init_eps=init, process_eps=eps, uniforms=us)
        with torch.no_grad():
            p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
            o = {k: (v[1:].contiguous().pin_memory() if host else v[1:].to(DEV)) for k, v in obs.items()}
            outs.append(p.forward_loop(observations=o, controls=controls[1:].to(DEV)))
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])


def test_forward_loop_cuda_graph_replay_matches_eager():
    """Small problems: the second forward_loop call with the same shapes captures the T-step recursion in a CUDA
    graph.  Same generator state -> same draws -> the replayed result equals the eager one."""
    name, sd, N, Mp, T = "PushCrossmodalParticleFilter", 2, 6, 30, 5
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=11)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    o = {k: v[1:].to(DEV) for k, v in obs.items()}
    c = controls[1:].to(DEV)
    p = fill_parameters(_product(name)(), seed=23).to(DEV).eval()
    p.num_particles = Mp
    outs = []
    with torch.no_grad():
        for call in range(4):  # 0: eager (first sight), 1: capture + replay, 2, 3: replay
            torch.manual_seed(1234)
            p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
            outs.append((p.forward_loop(observations=o, controls=c).clone(), p.particle_states.clone(),
                         p.particle_log_weights.clone()))
        assert p.__dict__["_mmf_loop_graph"]["graph"] not in (None, False), "the loop was not captured"
        p.graph_max_particles = 0
        torch.manual_seed(1234)
        p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
        eager = p.forward_loop(observations=o, controls=c)
    torch.cuda.synchronize()
    for est, st, lw in outs[2:]:
        assert torch.equal(est, outs[1][0]) and torch.equal(st, outs[1][1]) and torch.equal(lw, outs[1][2])
    assert torch.isfinite(outs[1][0]).all()
    # eager and replay consume the generator differently only if torch changes its graph-safe Philox bookkeeping;
    # the estimates agree statistically in any case, and bit for bit when the draws coincide
    assert_close(outs[0][0].cpu(), eager.cpu(), 1e-6, msg="eager twice")
    assert float((outs[1][0] - eager).abs().max()) < 1.0


def test_weight_gradients_are_bit_reproducible():
    """SURVEY.md section 7 hard part 4: the parameter-gradient reductions use no floating-point atomics (per-CTA partial
    sums + a fixed-order second pass), so repeated launches on the same inputs agree bit for bit -- at a row count that
    spreads over every CTA of the grid, and through a whole fused BPTT step."""
    K, L, P, sd = 2, 7, 8192 * 30, 2
    g = torch.Generator(device=DEV).manual_seed(5)
    act = torch.randn(K, L + 1, 16, P, 4, device=DEV, generator=g)
    delta = torch.randn(K, L + 1, 16, P, 4, device=DEV, generator=g)
    x = torch.randn(P, sd, device=DEV, generator=g)
    d_ll = torch.randn(K, P, device=DEV, generator=g)
    first = [t.clone() for t in ops.pf_heads_weight_grads(act, delta, x, d_ll)]
    for _ in range(3):
        again = ops.pf_heads_weight_grads(act, delta, x, d_ll)
        assert all(torch.equal(a, b) for a, b in zip(first, again))
    # fp32 reference of the reductions (chunk-major planes -> row matrices)
    A, D = ops.rows_view(act).double(), ops.rows_view(delta).double()
    assert_close(first[0].cpu(), torch.einsum("klpj,klpi->klji", D[:, :L], A[:, :L]).cpu(), 2e-4, msg="dW")
    assert_close(first[1].cpu(), D.sum(dim=2).cpu(), 2e-4, msg="db")
    del act, delta, A, D

    name, N, Mp, T = "PushCrossmodalParticleFilter", 64, 30, 4
    init, eps, _ = draw_noise(T, N, Mp, sd, seed=51)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=52)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    runs = []
    for _ in range(2):
        f = fill_parameters(_product(name)(), seed=53).to(DEV).train()
        f.num_particles = Mp
        f.noise = ReplayNoise(init_eps=init, process_eps=eps)
        for prm in f.dynamics_model.parameters():
            prm.requires_grad_(False)
        # the observation encoders are frozen here: cuDNN's convolution backward is outside this library's control
        for h in f.measurement_model.measurement_models:
            for prm in list(h.observation_image_layers.parameters()) if hasattr(h, "observation_image_layers") else []:
                prm.requires_grad_(False)
        for prm in f.measurement_model.crossmodal_weight_model.parameters():
            prm.requires_grad_(False)
        f.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
        est = f.forward_loop(observations={k: v[1:].to(DEV) for k, v in obs.items()}, controls=controls[1:].to(DEV))
        torch.mean((est - states[1:].to(DEV)) ** 2).backward()
        runs.append({k: q.grad.clone() for k, q in f.named_parameters() if q.grad is not None})
    assert len(runs[0]) > 20 and set(runs[0]) == set(runs[1])
    differing = [k for k in runs[0] if not torch.equal(runs[0][k], runs[1][k])]
    assert not differing, f"gradients differ between two identical runs: {differing[:5]}"


@pytest.mark.parametrize("rows", [1, 37, 4099])
def test_row_mlp_programs_match_torch_modules(rows):
    """mmf_row_mlp (one launch per per-trajectory stack) against the same modules evaluated by torch: observation
    encoders + concatenation of a head, PF / KF crossmodal weight models, virtual-sensor heads."""
    from multimodalfilter_b200.synthetic import synthetic_trajectories as synth

    _, obs, _ = synth(1, rows, 3, seed=61)
    o = {k: v[0].to(DEV) for k, v in obs.items()}
    cases = [
        ("head features", fill_parameters(M.PushCrossmodalParticleFilter(), seed=62).to(DEV).eval()),
        ("PF weights push", fill_parameters(M.PushCrossmodalWeightModel(know_image_blackout=False), seed=63).to(DEV).eval()),
        ("PF weights door", fill_parameters(M.DoorCrossmodalWeightModel(know_image_blackout=True), seed=64).to(DEV).eval()),
        ("KF weights", fill_parameters(M.DoorCrossmodalKalmanFilterWeightModel(state_dim=3), seed=65).to(DEV).eval()),
        ("virtual sensor door", fill_parameters(M.DoorVirtualSensorModel(), seed=66).to(DEV).eval()),
        ("virtual sensor push force", fill_parameters(M.PushVirtualSensorModel(modalities={"pos", "sensors"}), seed=67).to(DEV).eval()),
        ("virtual sensor push image", fill_parameters(M.PushVirtualSensorModel(modalities={"image"}), seed=68).to(DEV).eval()),
    ]
    for name, mod in cases:
        ops.PROFILE.reset(enabled=True)
        if name == "head features":
            plan = fused.PFPlan.build(mod)
            with torch.no_grad():
                got = [h.observation_features(o) for h in plan.heads]
            with torch.enable_grad():  # the torch-module path
                ref = [h.observation_features(o).detach() for h in plan.heads]
        else:
            with torch.no_grad():
                got = mod(observations=o)
            with torch.enable_grad():
                ref = mod(observations=o)
            got, ref = (list(got), [r.detach() for r in ref]) if isinstance(got, tuple) else ([got], [ref.detach()])
        assert "row_mlp" in ops.PROFILE.collect()["kernels"], f"{name}: mmf_row_mlp did not run"
        ops.PROFILE.reset()
        for g_, r_ in zip(got, ref):
            assert_close(g_.cpu(), r_.cpu(), 2e-5, msg=name)


@pytest.mark.parametrize("K,sd,rows", [(1, 3, 5), (2, 3, 1000), (3, 2, 257), (2, 1, 64)])
def test_kf_fuse_measurements_matches_the_reference_expressions(K, sd, rows):
    """R12 (mmf_kf_fuse_measurements) against the torch expressions of the reference's CrossmodalVirtualSensorModel /
    UnimodalVirtualSensorModel.forward (ref: crossmodal/base_models/crossmodal_kf.py:337-354, unimodal_kf.py:96-115)."""
    g = torch.Generator().manual_seed(71 + K + sd)
    z = torch.randn(K, rows, sd, generator=g)
    tril = torch.tril(torch.randn(K, rows, sd, sd, generator=g)) * 0.3
    tril.diagonal(dim1=-2, dim2=-1).abs_().add_(0.2)
    w = torch.rand(K, rows, sd, generator=g) + 0.05
    # crossmodal
    got_z, got_l = ops.kf_fuse_measurements(z.to(DEV), tril.to(DEV), w.to(DEV))
    ref_z, ref_cov = M._measurement_level(z, tril, w)
    assert_close(got_z.cpu(), ref_z, 1e-5, msg="crossmodal z")
    assert_close(got_l.cpu(), torch.linalg.cholesky(ref_cov), 1e-5, msg="crossmodal factor")
    # unimodal (the reference's arithmetic: elementwise reciprocal of the factors, float64 torch as the yardstick
    # because the matrix handed to inverse() holds K * 1e9 above its diagonal)
    got_z, got_c = ops.kf_fuse_measurements(z.to(DEV), tril.to(DEV), None)
    covs = tril @ tril.transpose(-1, -2)
    if K == 1:
        ref_z, ref_c = z[0], covs[0]
    else:
        prec = 1.0 / (tril + 1e-9)
        wd = torch.diagonal(prec, dim1=-2, dim2=-1)
        ref_z = M.weighted_average(z, wd)
        ref_c = torch.inverse((prec.sum(dim=0) + 1e-9).double()).float()
    assert_close(got_z.cpu(), ref_z, 1e-5, msg="unimodal z")
    assert_close(got_c.cpu(), ref_c, 1e-4, msg="unimodal covariance")


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
@pytest.mark.parametrize("name,M_,mode,estimation", [
    ("PushCrossmodalParticleFilter", 30, "multinomial", "weighted_average"),
    ("PushCrossmodalParticleFilter", 30, "systematic", "weighted_average"),
    ("PushCrossmodalParticleFilter", 30, None, "weighted_average"),       # training-style: no resampling
    ("PushCrossmodalParticleFilter", 17, "multinomial", "argmax"),
    ("PushUnimodalParticleFilter", 57, "multinomial", "argmax"),          # two particle chunks, ragged
    ("DoorCrossmodalParticleFilter", 128, "multinomial", "weighted_average"),  # four chunks, state_dim 3
    ("PushParticleFilter", 30, "multinomial_fast", "weighted_average"),
])
def test_one_launch_forward_loop_matches_the_per_step_kernels(name, M_, mode, estimation, precision):
    """F2: small problems run all T steps in ONE launch (k_pf_loop_small, a CTA per trajectory).  Its chain arithmetic is
    that of the fp32 per-step kernel (k_particle_chain_ffma) in the same order and its resampling IS nr_trajectory, so
    against the per-step path at precision fp32 on the same draws everything agrees bit for bit in the strict modes:
    estimates of every step, the final particle set, the final log-weights.  (The FAST modes' per-step path uses a
    different kernel with its own logits: agreement to rounding there.)  At precision bf16x3 / bf16 the one-launch kernel
    runs the layers on mma.sync with the same split bf16 operands as the tcgen05 per-step kernel: same products, another
    summation order, so agreement is to fp32 rounding (bf16: to the single-pass grade) with the odd resampling tie."""
    sd = 3 if name.startswith("Door") else 2
    N, T = 5, 7
    resample = mode is not None
    init, eps, us = draw_noise(T, N, M_, sd, seed=81, systematic=bool(mode and mode.startswith("systematic")))
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=82)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    o = {k: v[1:].to(DEV) for k, v in obs.items()}
    lib = _lib.load()
    if lib.mmf_pf_forward_loop_persistent(N, M_) != 1:
        assert M_ > 64 and lib.mmf_pf_forward_loop_persistent(N, 64) == 1 and lib.mmf_pf_forward_loop_persistent(N, 129) == 0
        pytest.skip("M > 64 takes the one-launch kernel only under MMF_PF_LOOP_SMALL=1 (tools/gpu scripts run that too)")
    outs = []
    for whole in (True, False):
        p = fill_parameters(_product(name)(), seed=83).to(DEV).eval()
        p.num_particles = M_
        p.precision = precision
        p.estimation_method = estimation
        p.resample = resample
        if resample:
            p.resample_mode = mode
        p.whole_loop = whole
        p.noise = ReplayNoise(init_eps=init, process_eps=list(eps), uniforms=list(us))
        ops.PROFILE.reset(enabled=True)
        with torch.no_grad():
            p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov)
            est = p.forward_loop(observations=o, controls=controls[1:].to(DEV))
        kernels = ops.PROFILE.collect()["kernels"]
        ops.PROFILE.reset()
        assert ("pf_forward_loop" in kernels) == whole, sorted(kernels)
        outs.append((est.clone(), p.particle_states.clone(), p.particle_log_weights.clone()))
    torch.cuda.synchronize()
    (e1, s1, l1), (e0, s0, l0) = outs
    assert torch.isfinite(e1).all()
    if precision != "fp32":
        tol = 2e-5 if precision == "bf16x3" else 3e-2
        scale = float(s0.abs().amax().clamp_min(1.0))
        differing = ((s1 - s0).abs().amax(dim=-1) > 10 * tol * scale).float().mean() if mode is not None else 0.0
        if estimation == "argmax" or precision == "bf16":  # a near-tie of two weights / a different draw moves an estimate
            close = ((e1 - e0).abs().amax(dim=-1) <= tol * e0.abs().amax().clamp_min(1.0)).float().mean()
            assert close > 0.9, f"only {float(close):.2f} of the estimates agree"
        else:
            assert_close(e1.cpu(), e0.cpu(), tol, msg="estimates")
            assert differing < 0.02, "more than a few resampling ties differ"
            if mode is None:
                assert_close(s1.cpu(), s0.cpu(), tol, msg="final particles")
                assert_close(l1.cpu(), l0.cpu(), tol, msg="final log-weights")
    elif mode == "multinomial_fast":
        assert_close(e1.cpu(), e0.cpu(), 1e-5, msg="estimates")
        assert (s1 != s0).any(dim=-1).float().mean() < 0.02, "more than a few resampling ties differ"
    else:
        assert torch.equal(e1, e0), f"estimates differ: max |d| = {float((e1 - e0).abs().max()):.3e}"
        assert torch.equal(s1, s0), "final particle states differ"
        assert torch.equal(l1, l0), "final log-weights differ"


@pytest.mark.parametrize("K,mask,with_w,M_", [(2, 0b11, True, 30), (2, 0b10, True, 30), (3, 0b101, False, 77), (1, 0b1, False, 1000)])
def test_reweight_train_kernels_match_torch_autograd(K, mask, with_w, M_):
    """mmf_pf_reweight_train_fwd / _bwd (training.Reweight: fusion over the enabled heads, reweight, normalise, estimate and
    their reverse mode) against the torch expressions of the training step and torch autograd, including a blacked-out
    modality (-inf weight) on some trajectories."""
    from multimodalfilter_b200 import training

    N, sd = 37, 2
    g = torch.Generator().manual_seed(91 + K + M_)
    ll = torch.randn(K, N, M_, generator=g) * 3.0
    modw = torch.randn(N, K, generator=g) if with_w else None
    on = [k for k in range(K) if (mask >> k) & 1]
    if with_w and len(on) > 1:
        modw[::5, on[0]] = -float("inf")  # quirk Q3: image blackout
    logw_in = torch.log_softmax(torch.randn(N, M_, generator=g), dim=1)
    states = torch.randn(N, M_, sd, generator=g)
    d_est = torch.randn(N, sd, generator=g)
    d_logw = torch.randn(N, M_, generator=g) * 0.1

    def run(fn, dev):
        a = ll.to(dev).double().requires_grad_() if dev == "cpu" else ll.to(dev).requires_grad_()
        w = None if modw is None else (modw.to(dev).double() if dev == "cpu" else modw.to(dev)).requires_grad_()
        li = (logw_in.to(dev).double() if dev == "cpu" else logw_in.to(dev)).requires_grad_()
        x = states.to(dev).double() if dev == "cpu" else states.to(dev)
        logw, est = fn(a, w, li, x)
        loss = (est * d_est.to(est)).sum() + (logw * d_logw.to(logw)).sum()
        loss.backward()
        return logw.detach().cpu(), est.detach().cpu(), a.grad.cpu(), None if w is None else w.grad.cpu(), li.grad.cpu()

    def torch_expr(a, w, li, x):  # the expressions of ParticleFilter._step_fused_train's torch path, in float64
        v = torch.stack([a[k] for k in on], dim=2)
        if w is not None:
            v = v + torch.stack([w[:, k] for k in on], dim=1)[:, None, :]
        u = li + torch.logsumexp(v, dim=2)
        ln = u - torch.logsumexp(u, dim=1, keepdim=True)
        return ln, torch.sum(torch.exp(ln)[:, :, None] * x, dim=1)

    ref = run(torch_expr, "cpu")
    got = run(lambda a, w, li, x: training.Reweight.apply(a, w, li, x, mask), DEV)
    names = ["logw", "estimate", "d_ll", "d_modality_logw", "d_logw_in"]
    for name, r, q in zip(names, ref, got):
        if r is None:
            assert q is None
            continue
        r = torch.nan_to_num(r.float(), nan=0.0)  # torch autograd: 0 * inf = nan on the blacked-out column; the kernel gives 0
        if name == "d_ll":
            off = [k for k in range(K) if k not in on]
            assert all(float(q[k].abs().max()) == 0.0 for k in off), "gradient leaked into a disabled head"
        assert_close(q, r, 2e-5, atol=1e-6, msg=name)


def test_forward_loop_with_long_trajectories():
    """M = 3000 particles per trajectory: normalise / resample goes through the multi-pass path (resample_big.cu), from the
    whole-sequence call and from the per-step path alike -- identical bits between the two, and the first step's estimate
    (no resampling upstream of it) within the bar of the oracle."""
    name, sd, N, Mp, T = "PushUnimodalParticleFilter", 2, 3, 3000, 3
    init, eps, us = draw_noise(T, N, Mp, sd, seed=95)
    states, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=96)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd)
    o = fill_parameters(getattr(port, name)(), seed=97).eval()
    o.num_particles = Mp
    o.noise = RecordedNoise(init_eps=init, process_eps=eps, uniforms=us, arithmetic="pinned")
    with torch.no_grad():
        o.initialize_beliefs(mean=states[0], covariance=cov)
        ref = o.forward_loop(observations={k: v[1:] for k, v in obs.items()}, controls=controls[1:])
    assert _lib.load().mmf_pf_resample_workspace_bytes(N, Mp) > 0
    outs = []
    for whole in (True, False):
        p = fill_parameters(_product(name)(), seed=97).to(DEV).eval()
        p.num_particles = Mp
        p.whole_loop = whole
        p.noise = ReplayNoise(init_eps=init, process_eps=list(eps), uniforms=list(us))
        with torch.no_grad():
            p.initialize_beliefs(mean=states[0].to(DEV), covariance=cov.to(DEV).contiguous())
            est = p.forward_loop(observations={k: v[1:].to(DEV) for k, v in obs.items()}, controls=controls[1:].to(DEV))
        outs.append((est.clone(), p.particle_states.clone(), p.particle_log_weights.clone()))
    torch.cuda.synchronize()
    (e1, s1, l1), (e0, s0, l0) = outs
    assert torch.equal(e1, e0) and torch.equal(s1, s0) and torch.equal(l1, l0)
    assert_close(e1[0].cpu(), ref[0], RTOL, msg="first-step estimate vs oracle")
    assert torch.isfinite(e1).all() and float((e1.cpu() - ref).abs().max()) < 0.5 * float(ref.abs().max())
