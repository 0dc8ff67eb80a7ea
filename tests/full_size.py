"""Helpers of the full-size kernel tests (test_training_full_size.py, test_inference_full_size.py,
test_kalman_full_size.py): the chain launchers' tile arithmetic restated, float64 evaluations of the packed chains, and
per-row error reports."""
import math

import torch

from util import U, kernel_ran

TILE, GROUPS = 128, 4        # k_particle_chain_ws / k_head_chain_bwd: rows per tile, groups (tiles in flight) per CTA


# ---- the launchers' arithmetic, restated ----------------------------------------------------------------------------
def chain_regime(P, sms):
    """k_particle_chain_ws / k_head_chain_bwd: ceil(tiles / 4) CTAs of 4 groups, at most one per SM; slot s covers tiles
    4 s .. 4 s + 3 and CTA u takes slots u, u + CTAs, ...  Returns the tiles of the busiest group, the tiles of the last
    slot (the issuer's `ng`), the rows of the last tile and the CTA count."""
    tiles = -(-P // TILE)
    slots = -(-tiles // GROUPS)
    ctas = min(slots, sms)
    return {"tiles": tiles, "ctas": ctas, "tiles_per_group": -(-slots // ctas),
            "last_slot": tiles - GROUPS * (slots - 1), "last_tile_rows": P - TILE * (tiles - 1)}


def nm_for_tiles(tiles, M, tile=TILE):
    """(N, M) with N M inside the last tile of `tiles` tiles of `tile` rows and not a multiple of `tile` (a ragged last
    tile)."""
    N = (tiles * tile - 1) // M
    assert (tiles - 1) * tile < N * M < tiles * tile
    return N, M


def profiled(fn, wants):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    for w in wants:
        assert kernel_ran(names, w), f"{w} did not run; kernels: {sorted(names)}"
    return out


# ---- float64 chains -------------------------------------------------------------------------------------------------
def _d(t):
    return t.detach().double()


def chain_layers(state, shared, feat_cols):
    """The 64x64 layers of a chain as (W (64, 64), b or None, kind) with kind RES_A / RES_B / MID, then the input and
    the output Linear.  feat_cols: the mid layer's state columns."""
    (in_lin, pre), (mid, post, out) = state, shared
    layers = []
    for r in pre:
        layers += [(_d(r.block1.weight), _d(r.block1.bias), "A"), (_d(r.block2.weight), _d(r.block2.bias), "B")]
    layers.append((_d(mid.weight[:, feat_cols]), None, "MID"))
    for r in post:
        layers += [(_d(r.block1.weight), _d(r.block1.bias), "A"), (_d(r.block2.weight), _d(r.block2.bias), "B")]
    return (_d(in_lin.weight), _d(in_lin.bias)), layers, (_d(out.weight), _d(out.bias))


def chain_forward(state, shared, feat_cols, x, rb, mid_relu, planes=None, preacts=None):
    """A whole chain in float64 on rows x (P, in_dim) with the hoisted mid-layer rows rb (P, 64): (P, out_dim).
    `planes`, a list, receives the input of every 64x64 layer and then that of the output layer (a tape's planes);
    `preacts`, a list, the input of every ReLU."""
    def relu(a):
        if preacts is not None:
            preacts.append(a)
        return torch.relu(a)

    (Wi, bi), layers, (Wo, bo) = chain_layers(state, shared, feat_cols)
    h = relu(x @ Wi.T + bi)
    res = None
    for W, b, kind in layers:
        if planes is not None:
            planes.append(h)
        if kind == "MID":
            h = h @ W.T + rb
            if mid_relu:
                h = relu(h)
        elif kind == "A":
            res, h = h, relu(h @ W.T + b)
        else:
            h = relu(h @ W.T + b + res)
    if planes is not None:
        planes.append(h)
    return h @ Wo.T + bo


def dynamics_moved(plan, states, eps, rowbias0, Mp):
    """x' = x + h[:sd] sigmoid(h[sd]) + q_tril eps through the float64 dynamics chain (mid layer linear)."""
    sd = plan.sd
    x = states.reshape(-1, sd).double()
    rb = rowbias0.double().repeat_interleave(Mp, dim=0)
    y = chain_forward(plan.dyn.state, plan.dyn.shared, slice(U, 2 * U), x, rb, mid_relu=False)
    q = plan.dyn.q()[: sd * sd].reshape(sd, sd).double().to(x.device)
    return x + y[:, :sd] * torch.sigmoid(y[:, sd:sd + 1]) + eps.double() @ q.T


def head_ll(spec, x, rb):
    """Log-likelihood of one measurement head (mid layer ReLU) in float64 for states x (P, sd) and rows rb (P, 64)."""
    return chain_forward(spec.state, spec.shared, slice(spec.feat_dim, spec.feat_dim + U), x, rb, mid_relu=True)[:, 0]


# ---- per-row errors -------------------------------------------------------------------------------------------------
def row_excess(got, ref, bar):
    """Worst |got - ref| / max(|ref|, rms(ref)) over the entries of each row, in units of `bar` (a number, or a tensor of
    one bar per row): (worst, its row).  A NaN in `got` counts as infinitely wrong."""
    got, ref = got.reshape(got.shape[0], -1).double(), ref.reshape(ref.shape[0], -1).double()
    scale = ref.pow(2).mean().sqrt()
    err = (got - ref).abs() / torch.maximum(ref.abs(), scale)
    per_row = torch.nan_to_num(err, nan=math.inf).amax(dim=1) / bar
    worst, row = per_row.max(dim=0)
    return float(worst), int(row)


def assert_rows(got, ref, bar, what, report, category, where=None):
    """row_excess within the bar; `report[category]` keeps the worst relative error.  `where(row)` names a failing row
    (default: its 128-row tile)."""
    worst, row = row_excess(got, ref, bar)
    bar_at = float(bar[row]) if torch.is_tensor(bar) else bar
    report[category] = max(report.get(category, 0.0), worst * bar_at)
    label = where(row) if where is not None else f"tile {row // TILE}"
    assert worst <= 1.0, f"{what}: {worst:.2f}x the bar {bar_at:g} at row {row} ({label})"
