"""Exchange kernels at ResNet-18 scale, bit for bit against the CPU golden model.

tests/test_gpu_kernels.py checks csrc/gossip.cu, gossip_dbuf.cu, ce_push.cu and sparse.cu on cnn2: 8 tensors,
20 tiles, grids of at most 6 CTAs.  The product runs them on the ResNet-18 arena (86 tensors, 8 569 tiles, single
tensors of 1 152 tiles, persistent grids of up to several hundred CTAs), where code paths run that cnn2 never reaches:
  - the tie look-back of sparse_compact_kernel walking more than one 32-tile window (tensors of more than 33 tiles);
  - histogram / candidate passes on a larger grid than the compaction (n_tiles > SP_MAX_OWN * grid);
  - tensors completed (claim_completed, cta_finish_tensors) after their tiles were spread over many CTAs;
  - the all-tie first spevent step (prev == theta_0, every key 0, tau == 0) on 1 152-tile tensors;
  - the per-warp push/mix pipeline with iters >> group_iters, and norm-on-write + trigger over 86 tensors.
Every case asserts the geometry it relies on, so that a model change cannot silently stop it from reaching its path.

R virtual ranks share one GPU (ops.local_world.LocalWorld).  The golden model (engine.simulator.RingSimulator) runs
on the CPU and is handed the kernels' own trigger decisions.  Gradients are drawn on the CPU from a seeded generator.
"""
from types import SimpleNamespace

import pytest
import torch

from eventgrad_b200.config import TrainConfig
from eventgrad_b200.engine.simulator import RingSimulator
from eventgrad_b200.models import build_model
from eventgrad_b200.parallel.arena import TILE
from eventgrad_b200.parallel.trigger import TriggerConfig

WINDOW = 32          # tiles per look-back iteration of sparse_compact_kernel (one per lane of the looking warp)
SP_MAX_OWN = 64      # csrc/sparse.cu: most tiles one CTA of the histogram / candidate passes takes


# ------------------------------------------------------------------------------------------------ CPU helpers
def lookback_depth(keys: torch.Tensor, k: int, tile: int = TILE) -> SimpleNamespace:
    """Recompute, for one fired tensor, what the tie look-back of sparse_compact_kernel does.

    `keys` are the tensor's |theta - prev| (fp32, its numel elements, before the send); `k` its top-k count.  The
    kernel selects every key > tau, where tau is the k-th largest key, plus the `need_eq` lowest-index keys == tau.
    A tile holding ties learns how many ties precede it by summing the per-tile tie counts of earlier tiles of the
    same tensor, 32 tiles per iteration, from the nearest down, until the start of the tensor or until need_eq
    earlier ties are found.  Returns
      tau      bit pattern of the k-th largest key (non-negative floats order like their bit patterns)
      need_eq  number of keys == tau that are selected
      ties     keys == tau per tile
      windows  look-back iterations per tile (0 for a tile without ties and for the tensor's first tile)
      depth    max(windows)
      deep     tiles whose look-back counts ties beyond its first window: their record slots are wrong if the
               look-back stops after one window
    """
    bits = keys.detach().float().contiguous().view(torch.int32).cpu()
    n = bits.numel()
    tau = int(torch.kthvalue(bits, n - k + 1).values)
    need_eq = k - int((bits > tau).sum())
    n_tiles = max(1, -(-n // tile))
    eq = torch.zeros(n_tiles * tile, dtype=torch.int64)
    eq[:n] = (bits == tau).long()
    ties = eq.view(n_tiles, tile).sum(1).tolist()
    before = [0]
    for q in ties:
        before.append(before[-1] + q)           # before[t] = ties in tiles [0, t)
    windows, deep = [], 0
    for t in range(n_tiles):
        w = pe = first = 0
        hi = t - 1
        if ties[t] > 0:
            while hi >= 0 and pe < need_eq:
                pe += before[hi + 1] - before[max(0, hi - WINDOW + 1)]
                hi -= WINDOW
                w += 1
                if w == 1:
                    first = pe
        windows.append(w)
        deep += pe > first
    return SimpleNamespace(tau=tau, need_eq=need_eq, ties=ties, windows=windows, depth=max(windows), deep=deep)


def test_lookback_depth_hand_built_layout():
    """tile = 4, 70 tiles, 278 keys: all 0 except element 5 (tile 1) = 1.0 and tile 50 = 2.0 (4 keys)."""
    keys = torch.zeros(278)
    keys[5] = 1.0
    keys[200:204] = 2.0
    # k = 5 + 160: tau = 0, need_eq = 160.  Ties per tile: tile 1 -> 3, tile 50 -> 0, tile 69 -> 2 (278 = 69*4 + 2)
    lb = lookback_depth(keys, 165, tile=4)
    assert lb.tau == 0 and lb.need_eq == 160
    assert lb.ties[0] == 4 and lb.ties[1] == 3 and lb.ties[50] == 0 and lb.ties[69] == 2 and sum(lb.ties) == 273
    assert lb.windows[0] == 0 and lb.windows[50] == 0           # first tile of the tensor; tile without ties
    assert set(lb.windows[1:33]) == {1}                         # one window reaches back to tile 0
    # tile 33: tiles 1..32 hold 127 < 160 ties, a second window reaches tile 0
    assert lb.windows[33] == 2 and lb.windows[69] == 2 and lb.depth == 2
    assert lb.deep == 69 - 33                                   # tiles 33..69 except 50
    # need_eq = 260: tile 64 reaches tile 0 after two windows (251 ties), tile 65 needs a third for tile 0
    lb = lookback_depth(keys, 265, tile=4)
    assert lb.need_eq == 260 and lb.windows[64] == 2 and lb.windows[65] == 3 and lb.depth == 3
    # distinct keys: tau unique, need_eq == 1; only the tile of tau looks back, and it finds no earlier tie
    keys = torch.arange(278, dtype=torch.float32) / 7
    lb = lookback_depth(keys, 278 - 150, tile=4)               # tau = key 150, in tile 37
    assert lb.tau == int(torch.tensor(150 / 7, dtype=torch.float32).view(torch.int32))
    assert lb.need_eq == 1 and lb.ties[37] == 1 and sum(lb.ties) == 1
    assert lb.windows[37] == 2 and lb.depth == 2 and lb.deep == 0


# ------------------------------------------------------------------------------------------------ GPU harness
def _cfg(algo, model="resnet18", **kw):
    base = dict(algo=algo, dataset="mnist" if model == "mlp" else "cifar10", model=model, lr=0.05, momentum=0.9,
                sync_mode="iter", horizon=1.0, thres_type=1, topk_percent=10.0)
    base.update(kw)
    return TrainConfig(**base).validate()


def _grid_cap(kind, R):
    """narrow: 16 CTAs per rank.  wide: the largest grid this one-GPU harness can host with all R grids co-resident
    and headroom for the other ranks' kernels (every wait is bounded by timeout_ns: a shortfall is status 1)."""
    if kind == "narrow":
        return 16
    from eventgrad_b200.ops import ext
    C = ext()
    return min(C.gossip_max_grid(0), C.gossip_dbuf_max_grid(0)) // (2 * R)


def _world(cfg, R, kind):
    from eventgrad_b200.ops.local_world import LocalWorld
    cap = _grid_cap(kind, R)
    w = LocalWorld(cfg, R, lambda: build_model(cfg.model), grid_cap=cap, timeout_ns=5_000_000_000)
    t = w.arenas[0].table
    G = w.backends[0].grid
    assert all(be.grid == G for be in w.backends)
    if kind == "narrow":
        assert t.n_tiles > SP_MAX_OWN * G          # sparse hist / cand passes get more CTAs than the compaction
    print(f"\n[grid] {cfg.model} {cfg.algo} R={R} {kind}: cap {cap} -> {G} CTAs per rank over {t.n_tiles} tiles")
    return w


def _resnet_geometry(t):
    assert t.n_tensors == 86 and max(t.tile_count) > SP_MAX_OWN     # tensors spread over several CTAs' ranges
    assert max(t.tile_count) > WINDOW + 1                            # a look-back can need a second window


def _pad_mask(t):
    m = torch.zeros(t.n_padded)
    for o, n in zip(t.offsets, t.numels):
        m[o:o + n] = 1
    return m


def _normal_grads(R, mask, gen, scale=0.05):
    return [torch.randn(mask.numel(), generator=gen) * scale * mask for _ in range(R)]


def _three_valued_grads(R, mask, gen):
    """-1/16, 0, +1/16: thousands of equal |theta - prev| keys per tensor, so tau sits inside big tie groups."""
    out = []
    for _ in range(R):
        u = torch.rand(mask.numel(), generator=gen)
        out.append(torch.where(u < 0.3, -0.0625, torch.where(u < 0.6, 0.0, 0.0625)) * mask)
    return out


def _high_precision_norms(theta, t):
    """fp64 per-tensor norms rounded to fp32.  (An fp32 CPU norm is off by up to ~3e-5 on 2.4 M elements.)"""
    return torch.stack([torch.linalg.vector_norm(theta[o:o + n].double()) for o, n in zip(t.offsets, t.numels)]).float()


def _check_theta(w, sim):
    torch.cuda.synchronize()
    for r, be in enumerate(w.backends):
        be.check_status()
        assert torch.equal(w.arenas[r].theta.cpu(), sim.theta[r]), f"rank {r} theta differs"
        assert float(w.arenas[r].grad.abs().max()) == 0.0, f"rank {r} grad not zeroed"


def _check_sparse(w, sim):
    _check_theta(w, sim)
    for r, be in enumerate(w.backends):
        for name in ("prev", "rep_l", "rep_r"):
            assert torch.equal(getattr(be, name).cpu(), getattr(sim, name)[r]), f"{name} rank {r}"
        assert be.num_events() == sim.events[r]
        assert be.bytes_sent() == sim.bytes[r]


def _spevent_steps(w, sim, grads, steps):
    """Step kernels and oracle side by side under the kernels' decisions.  Before every step, recompute each fired
    tensor's selection and look-back from the oracle's keys; after it, check tau and need_eq against what the kernel
    selected (sel_prefix / sel_remain).  Returns the look-back summaries of every step: [step][rank] {tensor: ...}."""
    t = sim.table
    hist = []
    for s in range(steps):
        fires = [be.fire.clone().bool().cpu() for be in w.backends]
        probe = [{i: lookback_depth((sim.theta[r][o:o + n] - sim.prev[r][o:o + n]).abs(), sim.k[i])
                  for i, (o, n) in enumerate(zip(t.offsets, t.numels)) if fires[r][i]} for r in range(w.world)]
        g = grads()
        w.step([x.cuda() for x in g])
        sim.step(g, fires=fires)
        torch.cuda.synchronize()
        for r, be in enumerate(w.backends):
            sel, rem = be.sel_prefix.cpu(), be.sel_remain.cpu()
            for i, lb in probe[r].items():
                assert (int(sel[i]), int(rem[i])) == (lb.tau, lb.need_eq), \
                    f"step {s + 1} rank {r} {t.names[i]}: kernel (tau, need_eq) differs from the oracle's keys"
        hist.append(probe)
    return hist


def _depths(hist):
    return [max((lb.depth for pr in step for lb in pr.values()), default=0) for step in hist]


# ------------------------------------------------------------------------------------------------ 1. dense
DENSE_MODES = {
    "dbuf": dict(),                                   # default: gossip_dbuf.cu, two inbox slots, no WAR ack
    "ack": dict(double_buffer=False),                 # gossip.cu single slot + ack
    "split": dict(overlap_push=True),                 # push phase kernel, then wait/mix/SGD phase
    "ce": dict(overlap_push=True, ce_push=True),      # copy-engine push (ce_push.cu), then wait/mix/SGD phase
}


@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["narrow", "wide"])
@pytest.mark.parametrize("R,mode", [(3, "dbuf"), (3, "ack"), (3, "split"), (3, "ce"), (2, "dbuf")])
def test_decent_resnet18_bitwise_vs_simulator(R, mode, grid):
    cfg = _cfg("decent", **DENSE_MODES[mode])
    w = _world(cfg, R, grid)
    t = w.arenas[0].table
    _resnet_geometry(t)
    for be in w.backends:
        assert (be.dbuf, be.overlap, be.ce_push) == (mode == "dbuf", mode in ("split", "ce"), mode == "ce")
        assert be.wire_dedup == (R == 2)               # 2-rank ring: theta crosses the link once
        assert -(-t.n_tiles // be.grid) > 8 * be.group_iters        # per-warp pipeline: iters >> depth
    sim = RingSimulator(R, w.arenas[0].theta.cpu(), t, "decent", lr=cfg.lr, momentum=cfg.momentum, serial_skip=False)
    mask, gen = _pad_mask(t), torch.Generator().manual_seed(1000 + R)
    for s in range(4):                                 # both inbox slots of the double-buffered kernel, twice
        g = _normal_grads(R, mask, gen)
        w.step([x.cuda() for x in g])
        sim.step(g)
    _check_theta(w, sim)
    w.close()


# ------------------------------------------------------------------------------------------------ 2. event
@pytest.mark.gpu
@pytest.mark.parametrize("grid", ["narrow", "wide"])
@pytest.mark.parametrize("R", [2, 3])
def test_event_resnet18_norms_decisions_bitwise(R, grid):
    """Free-running device FSM over 86 tensors: norm-on-write of 1 152-tile tensors, the decisions made from those
    norms, and the data path under them, every step against the oracle."""
    cfg = _cfg("event", horizon=0.95, initial_comm_passes=3)
    w = _world(cfg, R, grid)
    t = w.arenas[0].table
    _resnet_geometry(t)
    sim = RingSimulator(R, w.arenas[0].theta.cpu(), t, "event", TriggerConfig.from_train(cfg), lr=cfg.lr,
                        momentum=cfg.momentum)
    mask, gen = _pad_mask(t), torch.Generator().manual_seed(2000 + R)
    for s in range(8):
        fires = [be.fire.clone().bool().cpu() for be in w.backends]
        knorms = [be.cur_norm.cpu() for be in w.backends]           # norm-on-write of theta_k
        for r in range(R):
            torch.testing.assert_close(knorms[r], _high_precision_norms(sim.theta[r], t), rtol=3e-6, atol=1e-7,
                                       msg=lambda m: f"step {s + 1} rank {r} norms: {m}")
        g = _normal_grads(R, mask, gen)
        w.step([x.cuda() for x in g])
        sim.step(g, norms=knorms)
        for r in range(R):
            assert torch.equal(fires[r], sim.fire_history[-1][r]), f"step {s + 1} rank {r}: decisions differ"
    fired = torch.stack([f for step in sim.fire_history for f in step])
    assert fired.any() and not fired.all(), "thresholds no longer give mixed decisions"
    print(f"[event] fired per step (rank 0): {[int(step[0].sum()) for step in sim.fire_history]} of {t.n_tensors}")
    _check_theta(w, sim)
    for r, be in enumerate(w.backends):
        assert be.num_events() == sim.events[r]
        assert be.bytes_sent() == sim.bytes[r]
    w.close()


# ------------------------------------------------------------------------------------------------ 3. sparse top-k
@pytest.mark.gpu
@pytest.mark.parametrize("model,R,pct,grid", [("resnet18", 3, 10.0, "wide"), ("resnet18", 2, 1.0, "narrow"),
                                              ("resnet18", 3, 1.0, "narrow"), ("mlp", 3, 100.0, "wide"),
                                              ("mlp", 3, 1.0, "wide")])
def test_spevent_at_scale_bitwise_vs_simulator(model, R, pct, grid):
    cfg = _cfg("spevent", model=model, topk_percent=pct, initial_comm_passes=4, horizon=1.0)
    w = _world(cfg, R, grid)
    t = w.arenas[0].table
    if model == "resnet18":
        _resnet_geometry(t)
    else:
        assert max(t.tile_count) == 49                 # 784 x 128 weight: 49 tiles > one look-back window
    sim = RingSimulator(R, w.arenas[0].theta.cpu(), t, "spevent", TriggerConfig.from_train(cfg), lr=cfg.lr,
                        momentum=cfg.momentum, topk_percent=pct)
    mask, gen = _pad_mask(t), torch.Generator().manual_seed(3000 + R)
    hist = _spevent_steps(w, sim, lambda: _normal_grads(R, mask, gen), 5)
    # step 1: prev == theta_0, every key is 0 and ties: tau == 0, need_eq == k, the worst-case look-back
    for pr in hist[0]:
        assert len(pr) == t.n_tensors
        assert all(lb.tau == 0 and lb.need_eq == sim.k[i] for i, lb in pr.items())
    depths = _depths(hist)
    print(f"[spevent] {model} R={R} {pct}%: deepest look-back per step (windows of {WINDOW} tiles): {depths}")
    if pct >= 10.0:
        assert depths[0] > 1
    _check_sparse(w, sim)
    w.close()


# ------------------------------------------------------------------------------------------------ 4. tie look-back
@pytest.mark.gpu
@pytest.mark.parametrize("R,pct,grid", [(2, 37.0, "narrow"), (2, 10.0, "wide"), (3, 37.0, "wide"),
                                        (3, 10.0, "narrow")])
def test_spevent_tie_lookback_across_windows(R, pct, grid):
    """Three-valued gradients, momentum 0: after step 1 large groups of a tensor's keys are equal and spread over all
    of its tiles, so the ties at tau are counted over several 32-tile windows."""
    cfg = _cfg("spevent", topk_percent=pct, initial_comm_passes=3, horizon=1.0, momentum=0.0)
    w = _world(cfg, R, grid)
    t = w.arenas[0].table
    _resnet_geometry(t)
    sim = RingSimulator(R, w.arenas[0].theta.cpu(), t, "spevent", TriggerConfig.from_train(cfg), lr=cfg.lr,
                        momentum=0.0, topk_percent=pct)
    mask, gen = _pad_mask(t), torch.Generator().manual_seed(4000 + R)
    hist = _spevent_steps(w, sim, lambda: _three_valued_grads(R, mask, gen), 3)
    depths = _depths(hist)
    deep = [sum(lb.deep for pr in step for lb in pr.values()) for step in hist]
    print(f"[lookback] R={R} {pct}%: deepest look-back per step: {depths}; tiles counting ties beyond their first "
          f"window: {deep}")
    assert max(depths) >= 2
    # step 1 moves nothing (theta == prev), so a wrong tie set only shows from step 2 on: it must reach path 1 there
    assert any(d > 0 for d in deep[1:]), "no step after the first counts ties beyond one look-back window"
    _check_sparse(w, sim)
    w.close()
