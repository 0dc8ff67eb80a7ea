"""CPU-side checks of the product's host logic: the C ABI exports what the header declares, the
plan builder recognises the architectures, the packed layouts mean what include/mmf_b200.h says,
the API keeps the reference's assert-style error behaviour, and nothing silently runs on the CPU."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import multimodalfilter_b200 as mmf
from multimodalfilter_b200 import _lib, fused
from multimodalfilter_b200.crossmodal import models as M
from multimodalfilter_b200.synthetic import fill_parameters, synthetic_trajectories
from oracle.make_golden import REFERENCE, reference_available

from util import REPO, header_symbols, run_packed_chain, run_packed_rows


def test_shared_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    declared = header_symbols()
    assert len(declared) >= 16
    assert sorted(_lib.PROTOTYPES) == declared, "ctypes binding and header disagree"
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    missing = [s for s in declared if s not in exported]
    assert not missing, missing
    lib = ctypes.CDLL(_lib.LIB_PATH)  # loads without a GPU; no compute call is made here
    lib.mmf_abi_version.restype = ctypes.c_int
    assert lib.mmf_abi_version() == _lib.ABI_VERSION == 2


def test_library_contains_only_sm100a_code():
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = {tok for line in out.splitlines() for tok in line.replace(".", " ").split() if tok.startswith("sm_")}
    assert archs == {"sm_100a"}, archs


@pytest.mark.parametrize("name", ["PushCrossmodalParticleFilter", "DoorCrossmodalParticleFilter",
                                  "PushUnimodalParticleFilter", "PushParticleFilter", "DoorParticleFilter"])
def test_pf_plan_recognises_reference_architectures(name):
    task = "push" if name.startswith("Push") else "door"
    filt = M.MODEL_TYPES[task][name]()
    plan = fused.PFPlan.build(filt)
    assert plan is not None
    sd = filt.state_dim
    assert (plan.sd, plan.cd) == (sd, 7)
    if "Crossmodal" in name or "Unimodal" in name:
        assert plan.K == 2 and [h.feat_dim for h in plan.heads] == [64, 128]
        filt.measurement_model._enabled_models = [False, True]  # scripts poke the private list (train_push.py:157)
        assert plan.enabled_mask() == 0b10
    else:
        assert plan.K == 1 and plan.heads[0].feat_dim == 192 and plan.enabled_mask() == 1


def test_unknown_architecture_is_not_fused():
    class Odd(M.PushDynamicsModel):
        _mmf_fusable = False

    Odd.__name__ = "SomethingElse"
    filt = M.PushParticleFilter()
    filt.dynamics_model = Odd()
    assert fused.PFPlan.build(filt) is None


@pytest.mark.parametrize("dyn_cls", [M.PushDynamicsModel, M.DoorDynamicsModel, M.DoorDynamicsModelBrent])
def test_packed_dynamics_layout_matches_header(dyn_cls):
    dyn = fill_parameters(dyn_cls(), seed=3)
    spec = fused._DynamicsSpec(dyn)
    assert spec.ok
    chain, rows = spec.pack()
    sd = dyn.state_dim
    rng = np.random.default_rng(0)
    x = rng.standard_normal((9, sd)).astype(np.float32)
    u = rng.standard_normal((9, 7)).astype(np.float32)
    rowbias = run_packed_rows(rows.numpy(), 7, True, u)
    y = run_packed_chain(chain.numpy(), (sd, 1, 0, 3, sd + 1), x, rowbias)
    gate = 1.0 / (1.0 + np.exp(-y[:, sd]))
    mine = x + y[:, :sd] * gate[:, None]
    with torch.no_grad():
        ref, tril = dyn(initial_states=torch.from_numpy(x), controls=torch.from_numpy(u))
    np.testing.assert_allclose(mine, ref.numpy(), rtol=1e-4, atol=1e-5)
    q = spec.q().reshape(4, 4)  # flat sd*sd prefix, row-major
    np.testing.assert_allclose(spec.q()[: sd * sd].reshape(sd, sd).numpy(), tril[0].numpy())
    assert q.numel() == 16


@pytest.mark.parametrize("mods", [{"image"}, {"pos", "sensors"}, {"image", "pos", "sensors"}])
def test_packed_head_layout_matches_header(mods):
    head = fill_parameters(M.DoorMeasurementModel(modalities=mods), seed=4)
    spec = fused._HeadSpec(head, 3)
    assert spec.ok and spec.feat_dim == 64 * len(mods)
    chain, rows = spec.pack()
    _, obs, _ = synthetic_trajectories(1, 5, 3, seed=5)
    obs0 = {k: v[0] for k, v in obs.items()}
    particles = torch.randn(5, 6, 3)
    with torch.no_grad():
        feats = spec.observation_features(obs0)
        ref = head(states=particles, observations=obs0)
    rowbias = run_packed_rows(rows.numpy(), spec.feat_dim, False, feats.numpy())
    y = run_packed_chain(chain.numpy(), (3, 1, 1, 2, 1), particles.reshape(-1, 3).numpy(), np.repeat(rowbias, 6, axis=0))
    np.testing.assert_allclose(y.reshape(5, 6), ref.numpy(), rtol=1e-4, atol=1e-5)


def test_state_dict_keys_match_reference_layout():
    keys = set(M.PushCrossmodalParticleFilter().state_dict())
    for k in ("dynamics_model.Q_scale_tril", "dynamics_model.shared_layers.0.weight",
              "dynamics_model.state_layers.2.block1.weight",
              "measurement_model.measurement_models.0.state_layers.2.block1.weight",
              "measurement_model.measurement_models.1.observation_sensors_layers.0.weight",
              "measurement_model.crossmodal_weight_model.fusion_layers.3.bias"):
        assert k in keys, k
    door = M.DoorCrossmodalKalmanFilter().state_dict()
    assert "filter_models.0.dynamics_model.Q_scale_tril" in door
    assert "filter_models.1.virtual_sensor_model.r_layer.2.block2.weight" in door
    assert "dynamics_model.Q_scale_tril_diag" in M.DoorParticleFilter().state_dict()


def test_reference_error_conventions():
    filt = M.PushCrossmodalParticleFilter()
    with pytest.raises(AssertionError):  # not initialised (A.3)
        filt(observations={}, controls=torch.zeros(2, 7))
    mm = filt.measurement_model
    with pytest.raises(AssertionError):  # ref: crossmodal/base_models/crossmodal_pf.py:79-82
        mm.enabled_models = [True]
    with pytest.raises(AssertionError):
        mm.enabled_models = [1, 0]
    with pytest.raises(AssertionError):
        filt.initialize_beliefs(mean=torch.zeros(3, 5), covariance=torch.zeros(3, 2, 2))
    filt.eval()
    assert filt.num_particles == 300  # quirk Q8
    filt.train()
    assert filt.num_particles == 30


def test_cpu_tensors_fail_loudly_instead_of_falling_back():
    filt = M.PushCrossmodalParticleFilter().eval()
    with pytest.raises(_lib.MMFError, match="no CPU fallback"):
        filt.initialize_beliefs(mean=torch.zeros(3, 2), covariance=torch.eye(2)[None].expand(3, 2, 2))
    with pytest.raises(_lib.MMFError):
        mmf.ops.fuse_loglik(torch.zeros(2, 3, 2))


def test_product_never_imports_the_oracle():
    import ast

    bad = []
    for root, _, files in os.walk(os.path.join(REPO, "multimodalfilter_b200")):
        for f in files:
            path = os.path.join(root, f)
            if f.endswith(".py"):
                for node in ast.walk(ast.parse(open(path).read())):
                    names = []
                    if isinstance(node, ast.Import):
                        names = [a.name for a in node.names]
                    elif isinstance(node, ast.ImportFrom):
                        names = [node.module or ""]
                    if any(n == "oracle" or n.startswith("oracle.") for n in names):
                        bad.append(path)
            elif f.endswith((".cu", ".cuh", ".h")):
                if any("#include" in line and "oracle" in line for line in open(path)):
                    bad.append(path)
    assert not bad, bad


def test_install_aliases_make_reference_imports_resolve():
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import multimodalfilter_b200 as mmf; mmf.install()\n"
        "import torchfilter, fannypack\n"
        "from fannypack.nn import resblocks\n"
        "import torchfilter.types as types\n"
        "assert torchfilter.filters.ParticleFilter.__module__.startswith('multimodalfilter_b200')\n"
        "reference = %r\n"
        "if reference:\n"
        "    sys.path.insert(1, reference)\n"
        "    import warnings; warnings.filterwarnings('ignore')\n"
        "    import crossmodal\n"
        "    from multimodalfilter_b200 import fused\n"
        "    f = crossmodal.push_models.PushCrossmodalParticleFilter()\n"
        "    assert fused.PFPlan.build(f) is not None\n"
        "    k = crossmodal.door_models.DoorCrossmodalKalmanFilter()\n"
        "    assert fused.EKFPlan.build(list(k.filter_models)) is not None\n"
        "print('OK')\n"
    ) % (REPO, REFERENCE if reference_available() else None)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "OK" in res.stdout, res.stderr[-3000:]


# ---- image-encoder operand images (layouts documented in include/mmf_b200.h) -----------------------------
def _bf16_pairs(buf, count):
    """uint8 tensor -> float32 values of `count` bf16 numbers"""
    return buf[: 2 * count].view(torch.bfloat16).float()


@pytest.mark.parametrize("cin,cout", [(32, 32), (32, 16), (16, 8)])
def test_conv3x3_operand_image_layout(cin, cout):
    """mmf_enc_conv3x3's w_image: bf16 [tap 9][cin/8][2 npad rows: hi then lo][8] + fp32 bias[npad]; hi + lo restores
    the fp32 weight to 2^-17 and padded rows are zero."""
    from multimodalfilter_b200 import ops

    torch.manual_seed(cin + cout)
    conv = torch.nn.Conv2d(cin, cout, 3, padding=1)
    npad = 32 if cout > 16 else 16
    img = ops.enc_pack_conv3x3(conv)
    n_w = 9 * (cin // 8) * 2 * npad * 8
    assert img.numel() == 2 * n_w + 4 * npad
    w = _bf16_pairs(img, n_w).reshape(9, cin // 8, 2, npad, 8)          # (tap, chunk, hi|lo, row, channel-in-chunk)
    rebuilt = (w[:, :, 0] + w[:, :, 1]).permute(2, 1, 3, 0).reshape(npad, cin, 3, 3)  # (row, cin, ky, kx)
    ref = conv.weight.detach()
    assert torch.allclose(rebuilt[:cout], ref, rtol=0, atol=float(ref.abs().max()) * 2 ** -16)
    assert rebuilt[cout:].abs().max() == 0 if cout < npad else True
    bias = img[2 * n_w:].view(torch.float32)
    assert torch.equal(bias[:cout], conv.bias.detach()) and (bias[cout:] == 0).all()


def test_conv3x3_dx_stacked_image_layout():
    """MMF_ENC_VARIANT=3: bf16 [dy 3][cin/8][6 npad rows: hi dx-1 | hi dx0 | hi dx+1 | lo dx-1 | lo dx0 | lo dx+1][8]."""
    from multimodalfilter_b200 import ops

    torch.manual_seed(3)
    conv = torch.nn.Conv2d(32, 16, 3, padding=1)
    cin, cout, npad = 32, 16, 16
    img = ops.enc_pack_conv3x3_dx(conv)
    n_w = 3 * (cin // 8) * 6 * npad * 8
    w = _bf16_pairs(img, n_w).reshape(3, cin // 8, 2, 3, npad, 8)       # (ky, chunk, hi|lo, kx, row, channel-in-chunk)
    rebuilt = (w[:, :, 0] + w[:, :, 1]).permute(3, 1, 4, 0, 2).reshape(npad, cin, 3, 3)
    ref = conv.weight.detach()
    assert torch.allclose(rebuilt[:cout], ref, rtol=0, atol=float(ref.abs().max()) * 2 ** -16)


def test_stem_and_trunk_weight_buffers():
    from multimodalfilter_b200 import ops
    from multimodalfilter_b200.crossmodal import models as M
    from multimodalfilter_b200.encoders import ImageEncoder

    enc = M.PushCrossmodalParticleFilter().measurement_model.measurement_models[0].observation_image_layers
    assert isinstance(enc, ImageEncoder)
    convs = enc._trunk()
    assert convs is not None and [c.out_channels for c in convs] == [32, 32, 32, 16, 8]
    stem = ops.enc_pack_stem(convs[0])
    assert stem.shape == (25 * 32 + 32,)
    assert torch.equal(stem[: 25 * 32].reshape(25, 32).t().reshape(32, 1, 5, 5), convs[0].weight.detach())
    # the spanning-average-pool variant of the encoder is not the fused architecture: plain torch path
    pooled = M._image_encoder(64, spanning_avg_pool=True)
    assert pooled._trunk() is None
    # on CPU tensors / with autograd the module is the reference nn.Sequential
    y = enc(torch.zeros(2, 1, 32, 32))
    assert y.shape == (2, 64) and y.requires_grad


def test_chunk_major_rows_view_round_trip():
    """act / delta planes of the BPTT kernels: [column / 4][row][4] <-> (rows, 64)."""
    from multimodalfilter_b200 import ops

    rows = torch.arange(5 * 64, dtype=torch.float32).reshape(5, 64)
    planes = rows.reshape(5, 16, 4).transpose(0, 1).contiguous()        # (16, 5, 4)
    assert torch.equal(ops.rows_view(planes), rows)
    assert torch.equal(ops.rows_view(planes[None, None]), rows[None, None])


def test_row_programs_recycle_scratch_without_hazards():
    """fused.RowProgram recycles dead scratch slots (the per-row scratch lives in shared memory and decides the kernel's
    occupancy).  Executed symbolically here: every op must read values produced by the intended writer -- an input or an
    earlier op -- that no later op has overwritten in between, dst must not overlap src / res of its own op, and inputs
    must never sit in a recycled slot (all inputs are written before the first op runs)."""
    import numpy as np
    import torch

    from multimodalfilter_b200 import fused
    from multimodalfilter_b200.crossmodal import models as M

    def programs():
        m = M.DoorVirtualSensorModel()
        yield "door virtual sensor", m.encoded_program("sensor", [(m.shared_layers, None, m.units * len(m.modalities)),
                                                                    (m.z_layer, 0, m.units), (m.r_layer, m.units, m.units)]), m
        m = M.PushVirtualSensorModel(modalities={"pos", "sensors"})
        yield "push virtual sensor", m.encoded_program("sensor", [(m.shared_layers, None, m.units * len(m.modalities)),
                                                                    (m.z_layer, 0, m.units), (m.r_layer, m.units, m.units)]), m
        m = M.DoorCrossmodalKalmanFilterWeightModel(state_dim=3)
        yield "KF weight model", m.encoded_program("weights", [(m.fusion_layers, None, 3 * 64)]), m
        m = M.PushCrossmodalWeightModel(know_image_blackout=False)
        yield "PF weight model", m.encoded_program("weights", [(m.fusion_layers, None, 3 * 64)]), m
        f = M.PushCrossmodalParticleFilter()
        for h in fused.PFPlan.build(f).heads:
            yield "head features", h._feature_program(), None

    for name, prog, _ in programs():
        assert prog is not None, name
        # numeric execution of the program on the host (numpy) against the slot-free evaluation of the same ops
        rng = np.random.default_rng(0)
        S = np.full(prog.scratch, np.nan)
        for slot, d in zip(prog.in_slots, prog.in_dims):
            assert np.isnan(S[slot:slot + d]).all(), f"{name}: two inputs share scratch"
            S[slot:slot + d] = rng.standard_normal(d)
        values = {}  # (slot, dim) -> the vector the most recent writer put there
        for slot, d in zip(prog.in_slots, prog.in_dims):
            values[(slot, d)] = S[slot:slot + d].copy()
        for j, (op, lin) in enumerate(zip(prog.ops, prog.params)):
            assert op.dst + op.out_dim <= op.src or op.src + op.in_dim <= op.dst, f"{name}: op {j} dst overlaps src"
            assert op.res < 0 or op.dst + op.out_dim <= op.res or op.res + op.out_dim <= op.dst, f"{name}: op {j} dst overlaps res"
            x = S[op.src:op.src + op.in_dim]
            assert not np.isnan(x).any(), f"{name}: op {j} reads scratch nobody wrote"
            W = lin.weight.detach().double().numpy()
            y = W @ x + lin.bias.detach().double().numpy()
            if op.res >= 0:
                r = S[op.res:op.res + op.out_dim]
                assert not np.isnan(r).any(), f"{name}: op {j} reads a residual nobody wrote"
                y = y + r
            if op.act == 1:
                y = np.maximum(y, 0.0)
            elif op.act == 2:
                y = 1.0 / (1.0 + np.exp(-y))
            S[op.dst:op.dst + op.out_dim] = y
        for slot, d in zip(prog.out_slots, prog.out_dims):
            assert not np.isnan(S[slot:slot + d]).any(), f"{name}: an output slot was never written"
    # and the numbers: the recycled program equals the torch modules it was compiled from (one case, CPU, float64)
    m = M.PushCrossmodalWeightModel(know_image_blackout=False).double()
    prog = m.encoded_program("check", [(m.fusion_layers, None, 3 * 64)])
    obs = {"gripper_pos": torch.randn(1, 3, dtype=torch.float64), "gripper_sensors": torch.randn(1, 7, dtype=torch.float64),
           "image": torch.randn(1, 32, 32, dtype=torch.float64)}
    with torch.no_grad():
        ins = [enc(obs["image"][:, None]) if mod == "image" else obs[fused.OBS_KEY[mod]] for mod, enc in m._encoder_list()]
        ref = m.fusion_layers(m.encode(obs))[0].numpy()
    S = np.zeros(prog.scratch)
    for slot, d, x in zip(prog.in_slots, prog.in_dims, ins):
        S[slot:slot + d] = x[0].numpy()
    for op, lin in zip(prog.ops, prog.params):
        y = lin.weight.detach().numpy() @ S[op.src:op.src + op.in_dim] + lin.bias.detach().numpy()
        if op.res >= 0:
            y = y + S[op.res:op.res + op.out_dim]
        y = np.maximum(y, 0.0) if op.act == 1 else (1.0 / (1.0 + np.exp(-y)) if op.act == 2 else y)
        S[op.dst:op.dst + op.out_dim] = y
    got = S[prog.out_slots[0]:prog.out_slots[0] + prog.out_dims[0]]
    assert np.allclose(got, ref, rtol=1e-10, atol=1e-12), np.abs(got - ref).max()
