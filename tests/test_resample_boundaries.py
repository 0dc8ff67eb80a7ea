"""Resampling at its decision boundaries.

Every resampling path searches the CDF with a cheap fp32 key and falls back to the exact threshold of the pinned predicate
(DESIGN.md section 5) only when a probed CDF entry lies within a few ulp of that key.  Random uniforms land there about
once in a million draws, so the tests here aim the draws AT the CDF steps: from the pinned CDF `c` of the very logits a
kernel resamples, T_k = float64(fl(c_k / total)) is the point where the pinned predicate of entry k flips; the draws are
T_k, its neighbouring doubles, the un-rounded c_k / total and the ends of [0, 1).  Indices must equal those of the C
restatement (oracle/pinned) bit for bit, on every path, at the shapes where the dispatch and the kernels change behaviour:

    k_resample_fast<NG>            FAST modes, hard resampling, M <= 2048 (NG = 1, 2, 4, 8)
    k_normalize_resample<false,32>  one warp per trajectory: strict modes at M <= 2048, every mode with soft resampling
    k_normalize_resample<false,256> one CTA per trajectory, shared memory (M_out > 8192, soft at M > 2048, N > 65535)
    k_normalize_resample<true,256>  the same with a global workspace (a trajectory too long for shared memory)
    k_big_search_gather            hard resampling at M > 2048, N <= 65535 (resample_big.cu)
    k_pf_loop_small                the one-launch filter loop (M <= 64)

Each case also checks with torch.profiler that the kernel it is meant for is the one that ran, so that a change of a
dispatch threshold cannot silently move a case onto another path.
"""
import math

import numpy as np
import pytest
import torch

from multimodalfilter_b200 import ops
from oracle import pinned

from util import kernel_ran as _kernel_ran

DEV = "cuda:0"
MODES = ["multinomial", "multinomial_fast", "systematic", "systematic_fast"]
ONE_MINUS = 1.0 - 2.0 ** -53  # the largest double below 1

FAST = {ng: f"k_resample_fast<{ng}>" for ng in (1, 2, 4, 8)}
WARP = "k_normalize_resample<false,32>"
CTA = "k_normalize_resample<false,256>"
CTA_WS = "k_normalize_resample<true,256>"
BIG = "k_big_search_gather"
BIG_EST = "k_big_norm_est"
LOOP = "k_pf_loop_small"
_FAMILIES = ("k_resample_fast", "k_normalize_resample", "k_big_", "k_pf_loop_small")


def _fast_ng(M):
    return 1 if M <= 256 else 2 if M <= 512 else 4 if M <= 1024 else 8


def _systematic(mode):
    return mode.startswith("systematic")


# ---- the tie constructor (numpy only) ---------------------------------------------------------------------------------
def pinned_cdf(logits, mode):
    """(N, M) fp32 logits -> the pinned (un-normalised) CDF, (N, M) fp32."""
    N = logits.shape[0]
    u = np.zeros(N) if _systematic(mode) else np.zeros((N, 1))
    _, cdf = pinned.resample(logits, u, mode, num_samples=1, return_cdf=True)
    return cdf


def tie_points(c, ks):
    """T_k = float64(fl(c_k / total)): the pinned predicate of entry k, fl(c_k / total) < u, is false at u = T_k and true
    at the next double above it."""
    c = np.asarray(c, np.float32)
    return (c[np.asarray(ks, np.int64)] / c[-1]).astype(np.float64)


def tie_values(c, ks):
    """Draws around the CDF steps ks of one trajectory: T_k, the doubles on either side of it, float64(c_k) / float64(total)
    (un-rounded: the fp32 key and the exact threshold disagree there), then 0, the smallest positive double and 1 - 2^-53.
    Interleaved per k, so that a prefix covers whole steps; every value lies in [0, 1)."""
    c = np.asarray(c, np.float32)
    t = tie_points(c, ks)
    raw = c[np.asarray(ks, np.int64)].astype(np.float64) / np.float64(c[-1])
    vals = np.stack([t, np.nextafter(t, -np.inf), np.nextafter(t, np.inf), raw], axis=1).reshape(-1)
    vals = np.concatenate([[0.0, 5e-324, ONE_MINUS], vals])
    return np.clip(vals, 0.0, ONE_MINUS)


def systematic_u0(t, S):
    """u0 in [0, 1) with (u0 + j) / S == t exactly in float64 for some draw j (one exact tie in the trajectory), or None.
    j = floor(t S), u0 = t S - j, nudged one ulp of u0 + j at a time (u0 = x - j is exact: x lies in [j, j + 1))."""
    candidates, up, down = [t * S], t * S, t * S
    for _ in range(8):
        up, down = np.nextafter(up, np.inf), np.nextafter(down, -np.inf)
        candidates += [up, down]
    for x in map(float, candidates):
        j = math.floor(x)
        if x < 0.0 or j >= S:
            continue
        u0 = x - j
        if (u0 + j) / S == t:
            return u0
    return None


def tie_targets(c, fast, rng, extra=(), n_random=64):
    """CDF entries to aim at, most telling first: the caller's, in the FAST modes every place where the blocked CDF dips
    (c_k > c_{k+1}) and the ends of 256-groups and 8-segments, then the ends and random entries."""
    M = c.size
    ks = [int(k) for k in extra if 0 <= k < M]
    if fast:
        dips = np.flatnonzero(c[1:] < c[:-1])
        seg = np.arange(7, M, 8)
        ks += dips.tolist() + (dips + 1).tolist() + np.arange(255, M, 256).tolist()
        ks += rng.permutation(seg)[:256].tolist()
    ks += [0, 1, M // 2, M - 2, M - 1] + rng.integers(0, M, n_random).tolist()
    return np.array([k for k in dict.fromkeys(ks) if 0 <= k < M], dtype=np.int64)


def tie_uniforms(logits, mode, S, rng, extra=()):
    """Draws for (N, M) logits that put ties into every trajectory: (N, S) for the multinomial modes (rows filled with
    tie_values of their own targets, at random positions, the rest random), (N,) u0 for the systematic ones (one exact
    tie per trajectory, targets rotating over the rows; the first rows also take u0 = 0 and the smallest positive u0)."""
    cdf = pinned_cdf(logits, mode)
    N, M = logits.shape
    fast = mode.endswith("_fast")
    if _systematic(mode):
        u0 = rng.random(N)
        for n in range(N):
            ks = tie_targets(cdf[n], fast, rng, extra)
            k = ks[(n * 7919) % len(ks)] if n >= 2 or N < 4 else None
            if k is None:
                u0[n] = [0.0, 5e-324][n]
                continue
            r = systematic_u0(tie_points(cdf[n], [k])[0], S)
            if r is not None:
                u0[n] = r
        return u0
    u = rng.random((N, S))
    for n in range(N):
        ks = tie_targets(cdf[n], fast, rng, extra)
        ks = np.concatenate([ks[n % N::N], ks]) if N > 1 else ks  # rows start from different targets
        vals = tie_values(cdf[n], ks)[:S]
        u[n, rng.permutation(S)[: vals.size]] = vals
    return u


def random_logits(N, M, rng, scale=3.0):
    """Gaussian logits with dead particles, one row of equal weights (integer CDF steps) and one with a wide spread."""
    lg = (rng.standard_normal((N, M)) * scale).astype(np.float32)
    if M > 8:
        lg[rng.random((N, M)) < 0.02] = -np.inf
        lg[:, 1] = 0.0
    if N > 2:
        lg[1] = -1.5
        lg[2] *= 4
    return lg


def test_tie_constructor_flips_the_pinned_index():
    """CPU: at u = T_k the pinned lower bound is k, at the next double above it k + 1, and below it still k (no fp32
    quotient lies between T_k's lower neighbour and T_k).  Checked at every entry whose quotient strictly separates the
    entries before it from those after it (then every probe order agrees), strict and FAST CDFs.  The systematic
    constructor must find an exact tie for at least 90 % of the trajectories."""
    rng = np.random.default_rng(0)
    for mode in MODES:
        N, M = 6, 1500
        logits = random_logits(N, M, rng)
        cdf = pinned_cdf(logits, mode)
        checked = 0
        for n in range(N):
            q = (cdf[n] / cdf[n, -1]).astype(np.float32)
            before = np.maximum.accumulate(np.concatenate([[-np.inf], q[:-1]]).astype(np.float64))
            after = np.minimum.accumulate(np.concatenate([q[1:], [np.inf]])[::-1].astype(np.float64))[::-1]
            ks = tie_targets(cdf[n], mode.endswith("_fast"), rng)
            ks = ks[(before[ks] < q[ks]) & (q[ks] < after[ks])]
            t = tie_points(cdf[n], ks)
            row = lambda u: pinned.resample(logits[n : n + 1], u[None], "multinomial_fast" if "fast" in mode else "multinomial")[0]
            assert np.array_equal(row(t), ks)
            assert np.array_equal(row(np.nextafter(t, np.inf)), np.minimum(ks + 1, M - 1))
            assert np.array_equal(row(np.nextafter(t, -np.inf)), ks)
            raw = row(tie_values(cdf[n], ks)[6::4])  # float64(c_k) / float64(total): k or k + 1
            assert np.all((raw == ks) | (raw == np.minimum(ks + 1, M - 1)))
            checked += ks.size
        assert checked >= 200
        if _systematic(mode):
            for S in (M, M - 1, 2 * M + 3, 37):
                tried = hits = 0
                for n in range(N):
                    for k in tie_targets(cdf[n], mode.endswith("_fast"), rng)[:40]:
                        t = tie_points(cdf[n], [k])[0]
                        if t >= 1.0:
                            continue
                        tried += 1
                        u0 = systematic_u0(t, S)
                        if u0 is None:
                            continue
                        draws = (u0 + np.arange(S, dtype=np.float64)) / S  # the pinned (and kernel) positions
                        assert 0.0 <= u0 < 1.0 and np.any(draws == t), (S, k, u0)
                        idx = pinned.resample(logits[n : n + 1], np.array([u0]), mode, num_samples=S)[0]
                        assert idx[np.flatnonzero(draws == t)[0]] == pinned.resample(
                            logits[n : n + 1], np.array([[t]]), mode.replace("systematic", "multinomial"))[0, 0]
                        hits += 1
                assert hits >= 0.9 * tried, f"S={S}: only {hits} of {tried} trajectories got an exact systematic tie"


# ---- GPU helpers ------------------------------------------------------------------------------------------------------
def profiled(fn, want):
    """Run fn under torch.profiler and assert that the kernel `want` ran and no resampling kernel of another path did."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert _kernel_ran(names, want), f"{want} did not run; kernels: {sorted(names)}"
    family = next(f for f in _FAMILIES if want.startswith(f))
    others = sorted(n for n in names if any(f in n for f in _FAMILIES) and family not in n)
    assert not others, f"expected only {want}, also ran: {others}"
    return out


def assert_indices(idx, logits, u, mode, S, what=""):
    ref = pinned.resample(logits, u, mode, num_samples=S)
    assert idx.shape == ref.shape
    bad = np.argwhere(idx != ref)
    assert not len(bad), (f"{what}: {len(bad)} / {idx.size} indices differ from the pinned arithmetic; first (n, j, got, "
                          f"want): {[(int(n), int(j), int(idx[n, j]), int(ref[n, j])) for n, j in bad[:5]]}")
    return ref


def run_indices(logits, u, mode, S, want):
    fn = lambda: ops.resample_indices(torch.from_numpy(logits).to(DEV), torch.from_numpy(u).to(DEV),
                                      mode=ops.RESAMPLE_MODES[mode], M_out=S)
    return profiled(fn, want).cpu().numpy()


def run_normalize_resample(states, logw, mode, S, want, rng, alpha=1.0, extra=()):
    """pf_normalize_resample on tie draws built from the logits the kernel itself reports (a first call with random
    draws yields them: they do not depend on the draws).  Checks indices, the gather and the per-particle log-weights."""
    N, M, sd = states.shape
    kw = dict(mode=ops.RESAMPLE_MODES[mode], alpha=alpha, M_out=S, want_debug=True)
    st, lw = torch.from_numpy(states).to(DEV), torch.from_numpy(logw).to(DEV)
    u_rand = rng.random(N) if _systematic(mode) else rng.random((N, S))
    logits = ops.pf_normalize_resample(st, lw, uniforms=torch.from_numpy(u_rand).to(DEV), **kw)["logits"].cpu().numpy()
    u = tie_uniforms(logits, mode, S, rng, extra)
    out = profiled(lambda: ops.pf_normalize_resample(st, lw, uniforms=torch.from_numpy(u).to(DEV), **kw), want)
    assert np.array_equal(out["logits"].cpu().numpy(), logits)
    out["u"] = u
    idx = out["idx"].cpu().numpy()
    assert_indices(idx, logits, u, mode, S, f"{mode} M={M} M_out={S}")
    gathered = torch.gather(torch.from_numpy(states), 1, torch.from_numpy(idx)[:, :, None].expand(N, S, sd))
    assert torch.equal(out["states"].cpu(), gathered)  # a gather moves bits
    lw_out = out["logw"].cpu()
    if alpha < 1.0:
        expect = torch.gather(out["logw_norm"].cpu() - out["logits"].cpu(), 1, torch.from_numpy(idx))
        assert torch.equal(lw_out, expect)
    else:  # -logf(M): one value, within an ulp of -log M
        v = float(lw_out[0, 0])
        assert torch.equal(lw_out, torch.full((N, S), v)) and abs(v + math.log(M)) <= np.spacing(np.float32(math.log(M)))
    return out, idx, logits


gpu = pytest.mark.gpu


def _expected(mode, M):
    """the kernel of hard resampling at M <= 2048, M_out <= 8192"""
    return FAST[_fast_ng(M)] if mode.endswith("_fast") else WARP


# ---- ties through the fast and warp kernels ---------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("M", [30, 256, 257, 512, 513, 1024, 1025, 2048])
def test_ties_fast_and_warp_kernels(mode, M):
    rng = np.random.default_rng(M)
    N = 16
    logits = random_logits(N, M, rng)
    u = tie_uniforms(logits, mode, M, rng)
    assert_indices(run_indices(logits, u, mode, M, _expected(mode, M)), logits, u, mode, M, "resample_indices")
    states = rng.standard_normal((N, M, 2)).astype(np.float32)
    logw = (random_logits(N, M, rng) - 5).astype(np.float32)
    run_normalize_resample(states, logw, mode, M, _expected(mode, M), rng)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_ties_cta_kernel_many_draws(mode):
    """M_out > 8192 leaves the warp kernel for the CTA kernel (strict modes); the FAST kernel keeps M <= 2048 at any
    M_out."""
    rng = np.random.default_rng(9)
    N, M, S = 6, 1000, 9000
    want = FAST[4] if mode.endswith("_fast") else CTA
    logits = random_logits(N, M, rng)
    u = tie_uniforms(logits, mode, S, rng)
    assert_indices(run_indices(logits, u, mode, S, want), logits, u, mode, S, "resample_indices")
    states = rng.standard_normal((N, M, 2)).astype(np.float32)
    run_normalize_resample(states, random_logits(N, M, rng) - 5, mode, S, want, rng)


@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("M,N,want", [(1000, 8, WARP), (3000, 4, CTA), (100000, 2, CTA_WS)])
def test_ties_soft_resampling(mode, M, N, want):
    """alpha < 1: the mixed logits go through the warp kernel (M <= 2048, also in the FAST modes, whose blocked CDF is
    not monotone), the CTA kernel in shared memory, or the CTA kernel on a global workspace."""
    rng = np.random.default_rng(M + 1)
    states = rng.standard_normal((N, M, 2)).astype(np.float32)
    run_normalize_resample(states, random_logits(N, M, rng) - 5, mode, M, want, rng, alpha=0.5)


# ---- ties through the multi-pass kernels of long trajectories ---------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("M", [2049, 4096, 4097, 8193, 100000, 1 << 20])
def test_ties_big_kernels(mode, M):
    """Chunks of 4096, the first strided coarse level (M = 8193: windows of 2), M = 2^20 where CDF entries are about an
    ulp apart and the near-tie walk is the common case; M_out = M, M - 1 and M + 4097 (one more search chunk)."""
    rng = np.random.default_rng(M)
    N = 8 if M <= 8193 else 2 if M <= 100000 else 1
    logits = random_logits(N, M, rng, scale=3.0 if M < 100000 else 1.0)
    for S in (M, M - 1, M + 4097):
        u = tie_uniforms(logits, mode, S, rng)
        assert_indices(run_indices(logits, u, mode, S, BIG), logits, u, mode, S, f"M_out={S}")


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_ties_beyond_the_grid_limit(mode):
    """N = 65536 > the 65535 rows of a grid's y dimension: the multi-pass path does not apply; the CTA kernel strides over
    the trajectories.  The first and the last trajectories are checked against the oracle, all are range-checked."""
    N, M = 65536, 2049
    rows = np.r_[0:8, N - 8 : N]
    g = torch.Generator(device=DEV).manual_seed(3)
    logits = torch.randn(N, M, device=DEV, generator=g) * 3
    rng = np.random.default_rng(4)
    lg_rows = logits[torch.from_numpy(rows).to(DEV)].cpu().numpy()
    u_rows = tie_uniforms(lg_rows, mode, M, rng)
    shape = (N,) if _systematic(mode) else (N, M)
    u = torch.rand(shape, device=DEV, dtype=torch.float64, generator=g)
    u[torch.from_numpy(rows).to(DEV)] = torch.from_numpy(u_rows).to(DEV)
    idx = profiled(lambda: ops.resample_indices(logits, u, mode=ops.RESAMPLE_MODES[mode], M_out=M), CTA)
    assert int(idx.min()) >= 0 and int(idx.max()) < M
    assert_indices(idx[torch.from_numpy(rows).to(DEV)].cpu().numpy(), lg_rows, u_rows, mode, M, "N = 65536")
    del logits, u, idx
    torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("mode", ["systematic", "systematic_fast"])
@pytest.mark.parametrize("M", [64, 2048, 4096, 1 << 20])
def test_closed_form_systematic_on_equal_weights(mode, M):
    """Equal weights, S = M = 2^k, u0 = 0: c_k = k + 1 exactly, every draw j / M sits exactly on the step of entry j - 1,
    and the pinned lower bound is [0, 0, 1, ..., M - 2]."""
    want = BIG if M > 2048 else _expected(mode, M)
    logits = np.full((2, M), -math.log(M), np.float32)
    logits[1] = 7.0
    u0 = np.zeros(2)
    expect = np.concatenate([[0], np.arange(M - 1)])
    idx = run_indices(logits, u0, mode, M, want)
    assert np.array_equal(idx, np.stack([expect, expect]))
    assert_indices(idx, logits, u0, mode, M)


# ---- dead-particle plateaus ---------------------------------------------------------------------------------------------
PLATEAUS = {
    # M: dead runs [start, end); the big path: a leading run across a 4096 chunk, runs of 40 (> the 32-step walk) across
    # coarse windows of 8 and a chunk boundary, a trailing run of 3000
    40000: [(0, 5000), (8192 - 20, 8192 + 20), (12288 - 37, 12288 + 3), (20001, 20041), (37000, 40000)],
    2000: [(0, 300), (500, 540), (1024 - 20, 1024 + 20), (1800, 2000)],
}


@gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("M", sorted(PLATEAUS))
def test_ties_at_dead_particle_plateaus(mode, M):
    """Equal CDF entries behind every run of dead particles; draws aimed at the entry just before each run (and at the
    first live one after the leading run).  Bit-exact indices, no dead particle drawn, exact gather."""
    rng = np.random.default_rng(M + 7)
    N = 6
    logw = (rng.standard_normal((N, M)) - 5).astype(np.float32)
    for a, b in PLATEAUS[M]:
        logw[:, a:b] = -np.inf
    starts = [a - 1 for a, _ in PLATEAUS[M] if a > 0] + [b for a, b in PLATEAUS[M] if a == 0]
    extra = sorted(set(starts) | {s + 1 for s in starts} | {s - 1 for s in starts})
    want = BIG if M > 2048 else _expected(mode, M)
    states = rng.standard_normal((N, M, 2)).astype(np.float32)
    out, idx, _ = run_normalize_resample(states, logw, mode, M, want, rng, extra=extra)
    _assert_live(idx, logw, out["u"], mode)
    u = tie_uniforms(logw, mode, M, rng, extra)  # resample_indices on the raw log-weights
    idx = run_indices(logw, u, mode, M, want)
    assert_indices(idx, logw, u, mode, M)
    _assert_live(idx, logw, u, mode)


def _assert_live(idx, logw, u, mode):
    """No dead particle is drawn, with two exceptions that the pinned definition itself makes: a draw of exactly 0 (the
    lower bound is entry 0, whatever its weight: fl(c_0 / total) < 0 is false even for c_0 = 0) and, in the FAST modes, a
    draw aimed at the first entry of an 8-segment inside a dead run: the blocked CDF re-associates the segment totals there
    (Kogge-Stone), so it can rise by an ulp although the weights in between are zero."""
    N, S = idx.shape
    draws = (u[:, None] + np.arange(S)) / S if _systematic(mode) else u
    dead = ~np.isfinite(logw[np.arange(N)[:, None], idx]) & (draws > 0.0)
    if mode.endswith("_fast"):
        dead &= idx % 8 != 0
    assert not dead.any(), f"{int(dead.sum())} draws picked a dead particle"


# ---- gather and outputs off the common shape -------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode,M,S,sd,want", [
    ("multinomial_fast", 257, 100, 1, FAST[2]),
    ("systematic_fast", 257, 600, 3, FAST[2]),
    ("multinomial_fast", 1023, 1500, 4, FAST[4]),
    ("systematic_fast", 31, 31, 1, FAST[1]),
    ("multinomial_fast", 2047, 2000, 3, FAST[8]),
    ("multinomial", 4097, 2000, 3, BIG),
    ("systematic", 4097, 9001, 1, BIG),
    ("multinomial_fast", 5001, 8193, 4, BIG),
    ("systematic_fast", 4097, 4096, 3, BIG),
])
def test_gather_and_outputs_off_the_common_shape(mode, M, S, sd, want):
    """state_dim 1, 3, 4 (the FAST kernel's scalar gather), odd M (its scalar loads), M_out above and below M: indices,
    the gathered states, log-weights -log M and the weighted-average estimate."""
    rng = np.random.default_rng(M * sd)
    N = 5
    states = rng.standard_normal((N, M, sd)).astype(np.float32)
    logw = random_logits(N, M, rng) - 5
    out, _, _ = run_normalize_resample(states, logw, mode, S, want, rng)
    lw = logw.astype(np.float64)
    w = np.exp(lw - lw.max(1, keepdims=True))
    est = np.einsum("nm,nmd->nd", w / w.sum(1, keepdims=True), states.astype(np.float64))
    err = np.abs(out["estimate"].cpu().numpy() - est)
    assert np.all(err <= 1e-4 * np.maximum(np.abs(est), np.sqrt(np.mean(est ** 2)))), f"estimate off by {err.max():.3e}"


# ---- arg max estimate: exact duplicates and near-ties ----------------------------------------------------------------
ARGMAX_PATHS = [
    ("multinomial_fast", 1000, 1000, FAST[4]),
    ("systematic_fast", 200, 200, FAST[1]),
    ("multinomial", 1000, 1000, WARP),
    ("none", 1000, 1000, WARP),
    ("systematic", 1000, 9000, CTA),
    ("multinomial", 3000, 3000, BIG),
    ("none", 12288, 12288, BIG_EST),
]


@gpu
@pytest.mark.parametrize("mode,M,S,want", ARGMAX_PATHS)
def test_argmax_estimate_first_index_on_ties(mode, M, S, want):
    """The arg-max estimate is the first arg max of the path's own normalised log-weights fl(l - lse): exact duplicates
    of the maximum in different lanes, warps and 4096-particle chunks, and near-ties 0.42 ... 3 ulp of lse apart with the
    smaller log-weight first (below half an ulp both normalise to -lse and the first one wins).  Against float64 the
    pick may differ only within 2 ulp of lse."""
    rng = np.random.default_rng(M + S)
    pairs = [(37, 70), (5, 37), (31, 32), (255, 256), (3, 300, 700), (M // 2, M - 1), (4095, 4096), (5000, 9000),
             (8191, 8192), (100, 12000)]
    pairs = [p for p in pairs if max(p) < M]
    gaps = [(0.42, 2, 5), (0.5, 2, 5), (0.9, 2, 5), (1.5, 2, 5), (3.0, 2, 5), (0.42, M // 3, M - 2), (0.9, 40, M - 40)]
    N = len(pairs) + len(gaps)
    logw = (-0.01 - 0.5 * rng.random((N, M))).astype(np.float32)
    for n, p in enumerate(pairs):
        logw[n, list(p)] = 0.0
    ulps = []
    for n, (g, a, b) in enumerate(gaps, start=len(pairs)):
        logw[n, b] = 0.0
        row = logw[n].astype(np.float64)
        lse = np.log(np.exp(row).sum())
        ulp = float(np.spacing(np.float32(lse)))
        logw[n, a] = np.float32(-g * ulp)
        ulps.append(ulp)
    states = rng.standard_normal((N, M, 2)).astype(np.float32)
    states[:, :, 0] = np.arange(M, dtype=np.float32)  # the estimate names its particle
    st, lw = torch.from_numpy(states).to(DEV), torch.from_numpy(logw).to(DEV)
    if mode == "none":
        call = lambda: ops.pf_normalize_resample(st, lw, estimation=ops.ESTIMATE_ARGMAX, want_debug=True)
    else:
        u = rng.random(N) if _systematic(mode) else rng.random((N, S))
        call = lambda: ops.pf_normalize_resample(st, lw, estimation=ops.ESTIMATE_ARGMAX, mode=ops.RESAMPLE_MODES[mode],
                                                 M_out=S, uniforms=torch.from_numpy(u).to(DEV), want_debug=True)
    out = profiled(call, want)
    est = out["estimate"].cpu().numpy()
    picked = est[:, 0].astype(np.int64)
    assert np.array_equal(est, states[np.arange(N), picked])
    own = np.argmax(out["logw_norm"].cpu().numpy(), axis=1)  # first index of the maximum
    assert np.array_equal(picked, own), f"picked {picked.tolist()}, first arg max of logw_norm {own.tolist()}"
    for n, p in enumerate(pairs):
        assert picked[n] == min(p), (n, p, picked[n])
    l64 = logw.astype(np.float64)
    l64 = l64 - np.log(np.exp(l64).sum(1, keepdims=True))
    ref = np.argmax(l64, axis=1)
    for n in range(len(pairs), N):
        if picked[n] != ref[n]:
            assert l64[n, ref[n]] - l64[n, picked[n]] <= 2 * ulps[n - len(pairs)], (n, picked[n], ref[n])
    if mode != "none":
        assert_indices(out["idx"].cpu().numpy(), out["logits"].cpu().numpy(), u, mode, S)


# ---- the one-launch filter loop on ties ----------------------------------------------------------------------------------
class _Replay:
    """Noise source of the product filter replaying pre-drawn tensors."""

    def __init__(self, init_eps, process_eps, uniforms):
        self._init, self._eps, self._u = init_eps, list(process_eps), list(uniforms)

    def init_eps(self, M, N, sd, like):
        return self._init

    def process_eps(self, rows, sd, like):
        return self._eps.pop(0)

    def resample_uniforms(self, N, S, like):
        return self._u.pop(0)

    def randperm(self, M):
        return torch.randperm(M)


@gpu
@pytest.mark.parametrize("mode", ["multinomial", "systematic"])
@pytest.mark.parametrize("Mp", [30, 64])
def test_one_launch_loop_on_ties(Mp, mode):
    """PushUnimodalParticleFilter, one fp32 step: tie draws built from the per-step path's logits, replayed through the
    per-step kernels and through the one-launch loop kernel (M = 30: its register path, M = 64: nr_trajectory<32>).  The
    final particle sets are equal bit for bit and are the gather of the pinned indices."""
    from multimodalfilter_b200.crossmodal import models
    from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories

    N, sd, T = 8, 2, 1
    g = torch.Generator().manual_seed(Mp)
    init = torch.randn(Mp, N, sd, generator=g)
    eps = [torch.randn(N * Mp, sd, generator=g)]
    truth, obs, controls = synthetic_trajectories(T + 1, N, sd, seed=Mp + 1)
    cov = (torch.eye(sd) * 0.1)[None].expand(N, sd, sd).to(DEV).contiguous()
    o = {k: v[1:].to(DEV) for k, v in obs.items()}

    def run(whole, uniforms):
        p = fill_parameters(models.PushUnimodalParticleFilter(), seed=Mp + 2).to(DEV).eval()
        p.num_particles, p.precision, p.resample, p.resample_mode, p.whole_loop = Mp, "fp32", True, mode, whole
        p.noise = _Replay(init, eps, [uniforms])
        p.debug = None if whole else {}
        with torch.no_grad():
            p.initialize_beliefs(mean=truth[0].to(DEV), covariance=cov)
            p.forward_loop(observations=o, controls=controls[1:].to(DEV))
        torch.cuda.synchronize()
        return p

    rng = np.random.default_rng(Mp)
    u_rand = torch.from_numpy(rng.random(N) if _systematic(mode) else rng.random((N, Mp)))
    logits = run(False, u_rand).debug["logits"].cpu().numpy()
    u = torch.from_numpy(tie_uniforms(logits, mode, Mp, rng))
    step = run(False, u)
    assert np.array_equal(step.debug["logits"].cpu().numpy(), logits)
    whole = profiled(lambda: run(True, u), LOOP)
    ref = pinned.resample(logits, u.numpy(), mode, num_samples=Mp)
    assert np.array_equal(step.debug["idx"].cpu().numpy(), ref)
    moved = step.debug["moved"].cpu()
    gathered = torch.gather(moved, 1, torch.from_numpy(ref)[:, :, None].expand(N, Mp, sd))
    assert torch.equal(step.particle_states.cpu(), gathered)
    assert torch.equal(whole.particle_states.cpu(), gathered), "one-launch particles differ from the per-step ones"
    assert torch.equal(whole.particle_log_weights, step.particle_log_weights)
