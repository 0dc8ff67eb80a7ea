"""The inference kernels at the sizes the headline configurations run (C3: PushUnimodalParticleFilter, N = 4096
trajectories x M = 1000 particles, 409,600 hoisted (step, trajectory) rows; C5: up to 2^20 particles per trajectory, in
tiles of 128 x 2^20 = 2^27 particle rows), against float64.

Every kernel below has a persistent loop that starts only above a few tens of thousands of rows:

    k_particle_chain_ws<4,2,false>  bf16x3 / bf16 eval chain: a group takes a second 128-row tile only above
                                    4 groups x SMs x 128 rows; fused reweight epilogue (running two-term log-sum-exp
                                    over the head phases in logw_out, modality log-weights, logw_in on the last head)
    k_particle_chain_ffma           fp32 chain: 256-row tiles, grid = min(tiles, SMs)
    k_traj_rows                     hoisted rows: a warp per (plane, trajectory) item, 1,184 CTAs x 8 warps per sweep
    k_row_mlp                       observation encoders, weight models, virtual sensors: a CTA runs passes of
                                    warps x 8 rows, at most 2 CTAs per SM

Every shape restates its launcher's grid arithmetic in Python, asserts the regime it is meant for before it runs, and
torch.profiler confirms the kernel that ran.  Outputs are prefilled with NaN and the kernels are called through the raw C
entry points: a row a kernel never writes fails the comparison.  References are float64 on the GPU, in chunks of at most
2^22 rows:

  * chain: moved states through the float64 dynamics chain; ll of each enabled head through the float64 head chain from
    the kernel's own moved states (so dynamics error does not leak into the heads); logw_unnorm = logw_in +
    logsumexp_k(ll_ref[k] + modw[:, k]) over the enabled heads, whose -inf pattern the kernel must reproduce exactly;
  * hoisted rows: the control encoder and the mid Linear's trajectory columns (fused.pack_rows) in float64;
  * row programs: the same modules copied to float64, evaluated on the program's own inputs.

Bars are those of the small tests: 1e-4 (fp32, bf16x3) and 3e-2 (bf16) for the chain, 2e-5 for the fp32 row kernels.  At
2^27 rows the expected maximum of the rounding error is about 1.2x what it is at C4's 245,760 rows (it grows like
sqrt(2 ln n)).  Measured on a B200 (1000 W power limit), worst over every case: bf16x3 moved 1.5e-5, ll 6.4e-5 (C3;
6.2e-5 at 2^27 rows), logw 5.2e-6; bf16 moved 8.5e-3, ll 1.9e-2, logw 2.2e-3; fp32 moved 6.4e-7, ll 2.0e-6, logw 3.6e-7;
hoisted rows 1.9e-6; row programs 2.3e-6.  A misplaced tile, trajectory, pass or modality weight is wrong by O(1).
"""
import copy
import ctypes as C
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from multimodalfilter_b200 import _lib, fused, ops  # noqa: E402
from multimodalfilter_b200.crossmodal import models as M  # noqa: E402
from multimodalfilter_b200.synthetic import fill_parameters  # noqa: E402

from full_size import (  # noqa: E402
    GROUPS, assert_rows, chain_regime, dynamics_moved, head_ll, nm_for_tiles, profiled)

DEV = "cuda:0"
U = _lib.UNITS
CHUNK = 1 << 22              # rows per float64 reference chunk
FFMA_TILE = 256              # k_particle_chain_ffma: rows (threads) per tile
C3_N, C3_M = 4096, 1000
C5_N, C5_M = 128, 1 << 20    # the largest particle tile of C5
WS = "k_particle_chain_ws<4,2,false>"
FFMA = "k_particle_chain_ffma"
RTOL_X3 = 1e-4               # fp32 and bf16x3 (test_predict_measure_matches_oracle_modules)
RTOL_BF16 = 3e-2
RTOL_ROWS = 2e-5             # k_traj_rows, k_row_mlp: fp32 FFMA in the reference's summation order
MODELS = {"push_uni": "PushUnimodalParticleFilter", "push": "PushCrossmodalParticleFilter",
          "door": "DoorCrossmodalParticleFilter"}


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _plan(model):
    # a seed per model: Push and Door share the shapes of their hoisted-row layers, so one seed would give them the same rows
    f = fill_parameters(getattr(M, MODELS[model])(), seed=73 + list(MODELS).index(model)).to(DEV).eval()
    plan = fused.PFPlan.build(f)
    plan.refresh(torch.device(DEV))
    return f, plan


def _sweeps(shape, prefix):
    k, r = (int(v) for v in shape[len(prefix):].split("+"))
    return k, r


# ---- the chain launchers' arithmetic, restated ----------------------------------------------------------------------
def ffma_regime(P, sms):
    """launch_particle_chain_ffma: 256-row tiles, grid = min(tiles, SMs), CTA b takes tiles b, b + grid, ..."""
    tiles = -(-P // FFMA_TILE)
    grid = min(tiles, sms)
    return {"tiles": tiles, "ctas": grid, "tiles_per_cta": -(-tiles // grid), "last_tile_rows": P - FFMA_TILE * (tiles - 1)}


def chain_shape(shape, sms):
    """c3, c5, sweepsK+R (ws kernel: tiles = 4 SMs K + R, ragged last tile) or ffmaK+R (ffma kernel: tiles = SMs K + R,
    ragged last tile)."""
    if shape == "c3":
        return C3_N, C3_M
    if shape == "c5":
        return C5_N, C5_M
    if shape.startswith("sweeps"):
        k, r = _sweeps(shape, "sweeps")
        return nm_for_tiles(GROUPS * sms * k + r, 37)
    k, r = _sweeps(shape, "ffma")
    return nm_for_tiles(sms * k + r, 37, tile=FFMA_TILE)


def assert_chain_regime(shape, precision, P, sms):
    if precision == "fp32":
        g = ffma_regime(P, sms)
        if shape == "c3":
            assert P == C3_N * C3_M and g["ctas"] == sms and g["tiles_per_cta"] >= 2, g
        else:
            k, r = _sweeps(shape, "ffma")
            assert g["tiles"] == sms * k + r and g["ctas"] == sms, g
            assert g["tiles_per_cta"] == k + 1 and 0 < g["last_tile_rows"] < FFMA_TILE, g
        return g
    g = chain_regime(P, sms)
    if shape in ("c3", "c5"):
        assert P == (C3_N * C3_M if shape == "c3" else C5_N * C5_M) and g["ctas"] == sms, g
        assert g["tiles"] > GROUPS * sms * 2 and g["tiles_per_group"] >= 2, g  # every group loops
    else:
        k, r = _sweeps(shape, "sweeps")
        assert g["tiles"] == GROUPS * sms * k + r and g["ctas"] == sms, g
        assert g["tiles_per_group"] == k + 1 and g["last_slot"] == r and 0 < g["last_tile_rows"] < 128, g
    return g


# ---- raw entry points with NaN-prefilled outputs -------------------------------------------------------------------
def predict_measure(plan, states, eps, rowbias, logw, modw, mask, precision):
    N, Mp, _ = states.shape
    nan = float("nan")
    moved = torch.full_like(states, nan)
    logw_out = torch.full_like(logw, nan)
    ll = torch.full((plan.K, N, Mp), nan, device=DEV)
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_pf_predict_measure, C.byref(plan.struct), N, Mp, _lib.ptr(states), _lib.ptr(eps),
                         _lib.ptr(rowbias), _lib.ptr(logw), _lib.ptr(modw), mask, ops.PRECISIONS[precision],
                         _lib.ptr(moved), _lib.ptr(logw_out), _lib.ptr(ll), _lib.stream_of(states)))
    return moved, logw_out, ll


def traj_rows(plan, controls, feats):
    N = controls.shape[0]
    arr = (C.c_void_p * _lib.MAX_HEADS)()
    for k, f in enumerate(feats):
        arr[k] = None if f is None else f.data_ptr()
        _lib.ptr(f)  # the device check of a buffer whose pointer travels in `arr`
    out = torch.full((1 + plan.K, N, U), float("nan"), device=DEV)
    lib = _lib.load()
    _lib.check(_lib.call(lib.mmf_pf_traj_rows, C.byref(plan.struct), N, _lib.ptr(controls), arr, _lib.ptr(out),
                         _lib.stream_of(controls)))
    return out


def row_mlp(prog, inputs):
    rows = inputs[0].shape[0]
    outs = [torch.full((rows, d), float("nan"), device=DEV) for d in prog.out_dims]
    n_ops, n_in, n_out = len(prog.ops), len(inputs), len(outs)
    lib = _lib.load()
    for x in inputs:
        _lib.ptr(x)
    _lib.check(_lib.call(lib.mmf_row_mlp, rows, (_lib.MlpOp * n_ops)(*prog.ops), n_ops, _lib.ptr(prog._weights(DEV)),
                         (C.c_void_p * n_in)(*[x.data_ptr() for x in inputs]), (C.c_int32 * n_in)(*prog.in_dims),
                         (C.c_int32 * n_in)(*prog.in_slots), n_in, (C.c_void_p * n_out)(*[o.data_ptr() for o in outs]),
                         (C.c_int32 * n_out)(*prog.out_dims), (C.c_int32 * n_out)(*prog.out_slots), n_out, prog.scratch,
                         _lib.stream_of(inputs[0])))
    return outs


# ---- a. mmf_pf_predict_measure against float64 ---------------------------------------------------------------------
def _chain_cases():
    cases = [("bf16x3", "push_uni", "c3", 0b11), ("bf16x3", "push_uni", "c5", 0b11)]
    cases += [("bf16x3", "push", s, m) for s in ("sweeps1+1", "sweeps2+2", "sweeps1+3") for m in (0b11, 0b01, 0b10)]
    cases += [("bf16x3", "door", "c3", 0b11), ("bf16", "push_uni", "c3", 0b11), ("bf16", "door", "sweeps2+2", 0b11)]
    cases += [("fp32", "push_uni", "c3", 0b11)]
    cases += [("fp32", m, s, mask) for m in ("push", "door") for s in ("ffma1+1", "ffma3+2") for mask in (0b11, 0b10)]
    return cases


def chain_references(plan, states, eps, rowbias, logw_in, modw, mask, moved):
    """float64 moved states (P, sd), ll (K, P) (NaN for disabled heads) and logw_unnorm (P,)."""
    N, Mp, sd = states.shape
    P, K = N * Mp, plan.K
    on = [k for k in range(K) if (mask >> k) & 1]
    x_in, x = states.reshape(P, sd), moved.reshape(P, sd).double()
    moved_ref = torch.empty(P, sd, dtype=torch.float64, device=DEV)
    ll_ref = torch.full((K, P), float("nan"), dtype=torch.float64, device=DEV)
    for a in range(0, P, CHUNK):
        b = min(P, a + CHUNK)
        n = torch.arange(a, b, device=DEV) // Mp
        moved_ref[a:b] = dynamics_moved(plan, x_in[a:b], eps[a:b], rowbias[0][n], 1)
        for k in on:
            ll_ref[k, a:b] = head_ll(plan.heads[k], x[a:b], rowbias[1 + k][n].double())
    terms = ll_ref[on].T
    if modw is not None:
        terms = terms + modw[:, on].double().repeat_interleave(Mp, dim=0)
    logw_ref = logw_in.reshape(P).double() + torch.logsumexp(terms, dim=1)
    return moved_ref, ll_ref, logw_ref


@pytest.mark.parametrize("precision,model,shape,mask", _chain_cases())
def test_predict_measure_matches_float64(precision, model, shape, mask):
    """mmf_pf_predict_measure at C3, C5's largest tile and constructed sweep counts: moved states, ll of every enabled
    head and the fused logw_unnorm against float64, worst error per row; logw's -inf pattern (dead particles, blacked-out
    heads) must equal the reference's; ll planes of disabled heads must stay NaN."""
    sms = _sms()
    N, Mp = chain_shape(shape, sms)
    P = N * Mp
    regime = assert_chain_regime(shape, precision, P, sms)
    f, plan = _plan(model)
    K, sd = plan.K, plan.sd
    g = torch.Generator(device=DEV).manual_seed(P + mask)
    states = torch.randn(N, Mp, sd, device=DEV, generator=g)
    eps = torch.randn(P, sd, device=DEV, generator=g)
    rowbias = torch.randn(1 + K, N, U, device=DEV, generator=g)
    logw_in = torch.log_softmax(torch.randn(N, Mp, device=DEV, generator=g), dim=1)
    logw_in[torch.rand(N, Mp, device=DEV, generator=g) < 0.01] = -math.inf  # dead particles
    modw = None
    if f.measurement_model.crossmodal_weight_model is not None:
        modw = torch.randn(N, K, device=DEV, generator=g)
        modw[::5, 0] = -math.inf  # quirk Q3: the image head blacked out
        modw[1, [k for k in range(K) if (mask >> k) & 1]] = -math.inf  # every enabled head of one trajectory
    moved, logw, ll = profiled(lambda: predict_measure(plan, states, eps, rowbias, logw_in, modw, mask, precision),
                               [FFMA if precision == "fp32" else WS])
    moved_ref, ll_ref, logw_ref = chain_references(plan, states, eps, rowbias, logw_in, modw, mask, moved)
    bar = RTOL_BF16 if precision == "bf16" else RTOL_X3
    report = {}
    assert_rows(moved.reshape(P, sd), moved_ref, bar, "moved states", report, "moved")
    for k in range(K):
        if (mask >> k) & 1:
            assert_rows(ll[k].reshape(P, 1), ll_ref[k, :, None], bar, f"head {k} ll", report, "ll")
        else:
            assert torch.isnan(ll[k]).all(), f"head {k} is disabled but its ll plane was written"
    got, dead = logw.reshape(P), torch.isneginf(logw_ref)
    assert not torch.isnan(logw_ref).any() and not torch.isposinf(logw_ref).any()
    assert bool(dead.any()), "the reference has no -inf row: the pattern check would be empty"
    wrong = torch.isneginf(got) != dead
    assert not wrong.any(), (f"logw_unnorm: {int(wrong.sum())} rows differ from the reference's -inf pattern, first "
                             f"{int(wrong.nonzero()[0])}")
    assert_rows(got[~dead, None], logw_ref[~dead, None], bar, "logw_unnorm", report, "logw")
    print(f"[{precision} {model} {shape} mask={mask:#04b}] P={P} {regime}: {int(dead.sum())} -inf rows; worst relative "
          "errors " + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- b. mmf_pf_traj_rows against float64 ---------------------------------------------------------------------------
TR_ITEMS = 148 * 8 * 8       # launch_traj_rows: at most 148 x 8 CTAs (fixed, not the SM count) of 8 warps, an item each


def _traj_rows_n(shape, planes):
    """c3: C3's hoisted T N = 409,600 rows; ragged: (1 + K) N = 9,472 k + r with k = 3 full sweeps and 0 < r < 9,472."""
    if shape == "c3":
        return 409600
    N = 3 * TR_ITEMS // planes + 1
    assert 3 * TR_ITEMS < planes * N < 4 * TR_ITEMS
    return N


@pytest.mark.parametrize("model,shape,missing", [("push", "c3", None), ("push", "ragged", None), ("door", "c3", None),
                                                 ("door", "ragged", None), ("push", "ragged", 0), ("door", "c3", 1)])
def test_traj_rows_match_float64(model, shape, missing):
    """mmf_pf_traj_rows over every (plane, trajectory) item against the float64 tensors fused.pack_rows packs: plane 0
    the control encoder then the mid Linear's control columns and bias, plane 1 + k head k's feature columns and bias.
    A head without features (`missing`) is skipped: its plane must stay NaN."""
    _, plan = _plan(model)
    K = plan.K
    N = _traj_rows_n(shape, 1 + K)
    items = (1 + K) * N
    sweeps = -(-items // TR_ITEMS)
    assert sweeps >= 4 and (shape == "c3" or items % TR_ITEMS != 0), (items, sweeps)
    g = torch.Generator(device=DEV).manual_seed(N + K)
    controls = torch.randn(N, plan.cd, device=DEV, generator=g)
    feats = [None if k == missing else torch.randn(N, h.feat_dim, device=DEV, generator=g) for k, h in enumerate(plan.heads)]
    out = profiled(lambda: traj_rows(plan, controls, feats), ["k_traj_rows"])
    d = lambda t: t.detach().double()  # noqa: E731
    enc_lin, enc_res = plan.dyn.control
    h = torch.relu(controls.double() @ d(enc_lin.weight).T + d(enc_lin.bias))
    for r in enc_res:
        t = torch.relu(h @ d(r.block1.weight).T + d(r.block1.bias))
        h = torch.relu(t @ d(r.block2.weight).T + d(r.block2.bias) + h)
    mid = plan.dyn.shared[0]
    report = {}
    assert_rows(out[0], h @ d(mid.weight[:, :U]).T + d(mid.bias), RTOL_ROWS, "control rows", report, "control")
    for k, spec in enumerate(plan.heads):
        if feats[k] is None:
            assert torch.isnan(out[1 + k]).all(), f"head {k} has no features but its plane was written"
            continue
        mid = spec.shared[0]
        ref = feats[k].double() @ d(mid.weight[:, :spec.feat_dim]).T + d(mid.bias)
        assert_rows(out[1 + k], ref, RTOL_ROWS, f"head {k} rows", report, "heads")
    print(f"[{model} {shape} missing={missing}] N={N}: {items} items, {sweeps} sweeps of {TR_ITEMS}; worst relative "
          "errors " + " ".join(f"{c} {v:.2e}" for c, v in report.items()))


# ---- c. mmf_row_mlp programs against float64 ------------------------------------------------------------------------
RM_ROWS, RM_WARPS, RM_TILE_BYTES = 8, 16, 2 * 64 * 64 * 4


def row_mlp_regime(scratch, rows, sms):
    """launch_row_mlp: warps per CTA from the shared-memory budget (one CTA per SM with the whole window, or two with half
    of it each, whichever holds more warps), warps x 8 rows per pass, at most SMs x CTAs-per-SM CTAs.  k_row_mlp has no
    static shared memory, so its window is the opt-in maximum."""
    window = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    per_warp = RM_ROWS * scratch * 4

    def fit(budget):
        return min(RM_WARPS, (budget - RM_TILE_BYTES - 1024) // per_warp) if budget > RM_TILE_BYTES + 1024 else 0

    w1, w2 = fit(window), fit(window // 2)
    per_sm = 2 if 2 * w2 >= w1 else 1
    warps = w2 if per_sm == 2 else w1
    cta_rows = warps * RM_ROWS
    passes = -(-rows // cta_rows)
    cap = sms * per_sm
    return {"warps": warps, "cta_rows": cta_rows, "cap": cap, "ctas": min(passes, cap),
            "min_passes_per_cta": passes // min(passes, cap), "last_pass_rows": rows - cta_rows * (passes - 1)}


def _encoded64(mod, inputs):
    """The concatenated encoder features of a float64 module, the image features taken from the program's input."""
    return torch.cat([x.double() if m == "image" else enc(x.double()) for (m, enc), x in zip(mod._encoder_list(), inputs)],
                     dim=1)


def _row_programs():
    """(name, program, float64 reference of its outputs from its inputs): the seven programs of
    test_row_mlp_programs_match_torch_modules."""
    out = []
    plan = fused.PFPlan.build(fill_parameters(M.PushCrossmodalParticleFilter(), seed=62).to(DEV).eval())
    spec = plan.heads[1]  # pos + sensors: the head whose features are a program (the image head has only the CNN)

    def features(ins, m=copy.deepcopy(spec.head).double()):
        return [_encoded64(m, ins)]

    out.append(("head features", spec._feature_program(), features))
    for name, mod, key in [
        ("PF weights push", M.PushCrossmodalWeightModel(know_image_blackout=False), "weights"),
        ("PF weights door", M.DoorCrossmodalWeightModel(know_image_blackout=True), "weights"),
        ("KF weights", M.DoorCrossmodalKalmanFilterWeightModel(state_dim=3), "weights"),
        ("virtual sensor door", M.DoorVirtualSensorModel(), "sensor"),
        ("virtual sensor push force", M.PushVirtualSensorModel(modalities={"pos", "sensors"}), "sensor"),
        ("virtual sensor push image", M.PushVirtualSensorModel(modalities={"image"}), "sensor"),
    ]:
        mod = fill_parameters(mod, seed=63 + len(out)).to(DEV).eval()
        m64 = copy.deepcopy(mod).double()
        if key == "weights":  # the calls of _PFWeights.forward / _KFWeights.raw
            prog = mod.encoded_program(key, [(mod.fusion_layers, None, 3 * U)])

            def ref(ins, m=m64):
                return [m.fusion_layers(_encoded64(m, ins))]
        else:  # the call of _VirtualSensor.forward
            prog = mod.encoded_program(key, [(mod.shared_layers, None, U * len(mod.modalities)), (mod.z_layer, 0, U),
                                             (mod.r_layer, U, U)])

            def ref(ins, m=m64):
                h = m.shared_layers(_encoded64(m, ins))
                return [m.z_layer(h[:, :U]), m.r_layer(h[:, U:])]
        out.append((name, prog, ref))
    return out


@pytest.mark.parametrize("rows", [409600 + 7, 3 * 37888 + 5])
def test_row_mlp_programs_match_float64(rows):
    """mmf_row_mlp at rows where every CTA runs at least three passes and the last pass is ragged, for the warp count the
    launcher picks for each program: every output row against the same modules in float64."""
    sms = _sms()
    g = torch.Generator(device=DEV).manual_seed(rows)
    report = {}
    with torch.no_grad():
        for name, prog, ref in _row_programs():
            q = row_mlp_regime(prog.scratch, rows, sms)
            assert rows > 3 * q["cap"] * q["cta_rows"] and q["min_passes_per_cta"] >= 3, (name, q)
            assert 0 < q["last_pass_rows"] < q["cta_rows"], (name, q)
            inputs = [torch.randn(rows, dim, device=DEV, generator=g) for dim in prog.in_dims]
            outs = profiled(lambda: row_mlp(prog, inputs), ["k_row_mlp"])
            refs = ref(inputs)
            assert len(outs) == len(refs)
            for i, (o, r) in enumerate(zip(outs, refs)):
                assert_rows(o, r, RTOL_ROWS, f"{name} output {i}", report, name)
            print(f"[rows={rows}] {name}: {q}")
    print(f"[rows={rows}] worst relative errors " + " ".join(f"{c}: {v:.2e}" for c, v in report.items()))
