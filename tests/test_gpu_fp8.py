"""SC_MODE_FP8: the throughput tower and head kernels with e4m3 operands.

Numerics (DESIGN.md section 3.6): the weights of every tensor-core layer are e4m3 (round to nearest even) with a
power-of-two scale per output channel, s = 2^ceil(log2(amax / 448)); the epilogue forms a = acc * s + bias and then
runs the bf16 mode's fp32 LayerNorm / SE / residual / ReLU; each layer's output is stored as e4m3 (round to nearest
even, saturated to +-448).  The SE layers park their LayerNorm output in bf16 and keep bf16 SE weights.  The kernels
are checked layer by layer against a float64 emulation of exactly that (test_gpu_layer_reference's, with the e4m3
format), and these tests check batch independence, the launch variants, the entry points, the drivers and the
end-to-end accuracy on the bench batch.
"""
import functools

import numpy as np
import pytest
import scb200

from test_gpu_bench_config import batch2048, net19  # noqa: F401  (fixtures)
from test_gpu_layer_reference import (  # noqa: F401  (fixtures)
    FP8, LAUNCH_VARIANTS, _batch, _engine as _engine_any, _eval, check_launch_variant, check_selfplay_arena_and_game,
    games, nets, run_heads, run_throughput_layers)

pytestmark = pytest.mark.gpu

_engine = functools.partial(_engine_any, mode=scb200.SC_MODE_FP8)


# ---- 1 / 2. every layer against float64, on all test nets -------------------------------------------------------
@pytest.mark.parametrize("tag", ["n2", "stress", "bn_se", "ln_nose", "bn_nose"])
def test_fp8_tower_layers(nets, games, monkeypatch, tag):  # noqa: F811
    boards = [0, 1, 2, 3, 127, 128, 329, 330, 331, 332] if tag in ("n2", "stress") else None
    run_throughput_layers(FP8, nets, games, monkeypatch, tag, (1, 6), boards)


@pytest.mark.parametrize("tag", ["n2", "stress", "bn_se", "ln_nose", "bn_nose"])
def test_fp8_heads_from_tower_buffers(nets, games, monkeypatch, tag):  # noqa: F811
    run_heads(FP8, nets, games, monkeypatch, tag)


def test_fp8_has_no_latency_kernel(nets, games, monkeypatch):  # noqa: F811
    import scb200

    e = _engine(nets["n2"][1], monkeypatch, max_batch=16)
    try:
        pos, _, _ = _batch(games, 1)
        with pytest.raises(scb200.SCError):
            e.debug_tower(pos, 1, 1)
    finally:
        e.close()


# ---- 3. batch independence and launch variants ------------------------------------------------------------------
def test_fp8_rows_do_not_depend_on_the_batch(net19, batch2048, monkeypatch):  # noqa: F811
    """a leaf's priors and value are the same bits at n = 1, 37, 129 and 2048 (every size runs the throughput
    kernels; n <= 128 uses the fused value tail, larger batches the stand-alone one)"""
    games, pos, moves, off, mv_all, lp, v, pri_ref = batch2048
    e = _engine(net19[1], monkeypatch, max_batch=2048)
    try:
        full = e.eval(pos, moves, off)
        full = (full[0].copy(), full[1].copy())
        for n in (1, 37, 129):
            for s in (0, 1000):
                o = off[s:s + n + 1] - off[s]
                p, val = e.eval(pos[s:s + n], moves[off[s]:off[s + n]], o)
                assert np.array_equal(p, full[0][off[s]:off[s + n]]) and np.array_equal(val, full[1][s:s + n]), (n, s)
    finally:
        e.close()


@pytest.mark.parametrize("env", LAUNCH_VARIANTS)
def test_fp8_launch_variants_bit_identical(net19, batch2048, monkeypatch, env):  # noqa: F811
    check_launch_variant(scb200.SC_MODE_FP8, net19, batch2048, monkeypatch, env)


# ---- 4. entry points and drivers --------------------------------------------------------------------------------
def _eval_rows(e, moves, counts, pos):
    """sc_eval of packed leaves with the moves predict returned -> per-leaf (priors, value) for non-terminal leaves"""
    live = np.nonzero(counts > 0)[0]
    flat = np.concatenate([moves[i, :counts[i]] for i in live])
    off = np.concatenate(([0], np.cumsum(counts[live]))).astype(np.int32)
    pri, val = e.eval(pos[live], flat, off)
    return live, pri.copy(), val.copy(), off


def _random_game(rng, max_plies):
    import scb200

    h = []
    for _ in range(rng.randint(0, max_plies + 1)):
        mv = scb200.rules_probe(h)[0]
        if len(mv) == 0:
            break
        h.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
    return h


def test_fp8_predict_path_and_evaluator_equal_eval(nets, monkeypatch):  # noqa: F811
    """sc_predict_path and an sc_evaluator on an fp8 engine return exactly what sc_eval returns for the same packed
    leaves and legal moves"""
    import scb200

    rng = np.random.RandomState(5)
    gs = [_random_game(rng, 60) for _ in range(24)]
    roots, paths = [g[: len(g) // 2] for g in gs], [g[len(g) // 2:] for g in gs]
    e = _engine(nets["n2"][1], monkeypatch, max_batch=64)
    try:
        e.set_roots(roots)
        moves, counts, pri, val, pos = e.predict_path(np.arange(len(roots)), paths, positions=True)
        moves, counts, pri, val = moves.copy(), counts.copy(), pri.copy(), val.copy()
        live, ep, ev, off = _eval_rows(e, moves, counts, pos)
        assert len(live) > 0
        for k, i in enumerate(live):
            assert np.array_equal(pri[i, :counts[i]], ep[off[k]:off[k + 1]]) and val[i] == ev[k], i
    finally:
        e.close()
    e = _engine(nets["n2"][1], monkeypatch, max_batch=64)
    evl = scb200.Evaluator(e, 4)
    try:
        for i, (r, p) in enumerate(zip(roots, paths)):
            evl.set_root(i % 4, r)
            mv, cnt, pr, v = evl.predict(i % 4, p)
            assert cnt == counts[i] and np.array_equal(mv[:cnt], moves[i, :cnt]), i
            assert np.array_equal(pr[:cnt], pri[i, :cnt]) and v == val[i], i
    finally:
        evl.close()
        e.close()


def test_fp8_selfplay_arena_and_game(co, nets, monkeypatch):  # noqa: F811
    check_selfplay_arena_and_game(scb200.SC_MODE_FP8, co, nets, monkeypatch)


# ---- 5. accuracy on the bench batch -----------------------------------------------------------------------------
def _accuracy(p, v, pri_ref, v_ref, off):
    d = np.abs(p - pri_ref)
    tv, top = [], []
    for i in range(len(off) - 1):
        a, b = off[i], off[i + 1]
        if b > a:
            tv.append(0.5 * float(d[a:b].sum()))
            top.append(np.argmax(p[a:b]) == np.argmax(pri_ref[a:b]))
    return {"max_d_prior": float(d.max()), "mean_d_prior": float(d.mean()), "mean_tv": float(np.mean(tv)),
            "max_d_value": float(np.abs(v - v_ref).max()), "mean_d_value": float(np.abs(v - v_ref).mean()),
            "top_move_agreement": float(np.mean(top))}


# end-to-end gates, set from the first measured run on the 2048-leaf bench batch (max |d prior| 0.092, mean total-
# variation distance 0.046, max |d value| 0.089, top move agreeing on 84.2 % of the leaves) with a margin of about 1.5x
FP8_GATE = {"max_d_prior": 0.14, "mean_tv": 0.07, "max_d_value": 0.13, "top_move_agreement": 0.76}


def test_fp8_bench_workload_accuracy(net19, batch2048, monkeypatch):  # noqa: F811
    """19 blocks, 2048 random-play leaves against the fp32 oracle, printed next to bf16 and fp16 on the same batch"""
    import scb200

    games, pos, moves, off, mv_all, lp, v, pri_ref = batch2048
    res = {}
    for name, mode in (("fp8", scb200.SC_MODE_FP8), ("bf16", scb200.SC_MODE_BF16), ("fp16", scb200.SC_MODE_FP16)):
        p, val = _eval(net19[1], monkeypatch, pos, moves, off, mode=mode)
        assert np.isfinite(p).all() and np.isfinite(val).all()
        res[name] = _accuracy(p, val, pri_ref, v, off)
        print(name, {k: "%.4g" % x for k, x in res[name].items()})
    r = res["fp8"]
    assert r["max_d_prior"] <= FP8_GATE["max_d_prior"] and r["mean_tv"] <= FP8_GATE["mean_tv"]
    assert r["max_d_value"] <= FP8_GATE["max_d_value"] and r["top_move_agreement"] >= FP8_GATE["top_move_agreement"]
