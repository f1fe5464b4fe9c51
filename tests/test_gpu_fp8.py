"""SC_MODE_FP8: the throughput tower and head kernels with e4m3 operands.

Numerics (DESIGN.md section 3.6): the weights of every tensor-core layer are e4m3 (round to nearest even) with a
power-of-two scale per output channel, s = 2^ceil(log2(amax / 448)); the epilogue forms a = acc * s + bias and then
runs the bf16 mode's fp32 LayerNorm / SE / residual / ReLU; each layer's output is stored as e4m3 (round to nearest
even, saturated to +-448).  The SE layers park their LayerNorm output in bf16 and keep bf16 SE weights.  These tests
emulate exactly that in float64, layer by layer, and check batch independence, the launch variants, the entry points,
the drivers and the end-to-end accuracy on the bench batch.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_bench_config import batch2048, net19  # noqa: F401  (fixtures)
from test_gpu_fp16 import _eval, _engine as _engine_any, _u16_to_f64
from test_gpu_layer_reference import (  # noqa: F401  (fixtures and dtype-free helpers)
    PLANES, X, T, Y, BIT_EQUAL_MIN, _batch, _layers, _norm, _nhwc_to_nchw, _ulp_bf16, _bf16, games, nets)

pytestmark = pytest.mark.gpu

E4M3_MAX = 448.0


# ---- e4m3 arithmetic of the reference ---------------------------------------------------------------------------
def _rnd8(t):
    """round to e4m3 (nearest even), saturating at +-448 (cvt.rn.satfinite)"""
    return t.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(torch.float64)


def _ulp8(v):
    """Spacing of e4m3 numbers at |v|: 2^(e - 4) for normal numbers (|v| >= 2^-6), 2^-9 below (0 at 0)."""
    m, e = np.frexp(np.abs(v))
    return np.where(v == 0, 0.0, np.ldexp(1.0, np.maximum(e - 4, -9)))


def _scaled_weight(w):
    """[cout, ...] fp32 weights -> the engine's e4m3 weights times their per-output-channel power-of-two scale,
    float64: per channel s = 2^ceil(log2(amax / 448)) (1 when all zero), then e4m3(w / s) * s"""
    w = w.double()
    amax = w.abs().reshape(w.shape[0], -1).amax(dim=1).numpy()
    m, e = np.frexp(amax)
    s = np.where(amax > 0, np.ldexp(1.0, np.where(m <= 0.875, e - 9, e - 8)), 1.0)
    s = torch.from_numpy(s).reshape((-1,) + (1,) * (w.dim() - 1))
    return _rnd8(w / s) * s


def _conv_bias(sd, conv, x):
    w = _scaled_weight(sd[conv + ".weight"])
    return F.conv2d(x, w, sd[conv + ".bias"].double(), padding=w.shape[-1] // 2)


def _layer_reference(sd, layer, inp, resid):
    """One layer in float64 on the kernel's e4m3 inputs -> (out before the final rounding, z, gate, a = conv + bias).
    The SE layers' z is parked in bf16 and their SE weights are bf16, as in bf16 mode."""
    conv, norm, _, _, relu, se = layer
    a = _conv_bias(sd, conv, inp)
    z = _norm(sd, norm, a)
    if se is None:
        return (z.clamp_min(0) if relu else z), None, None, a
    if se == "residual":
        gate = torch.ones(z.shape[0], z.shape[1], 1, 1, dtype=torch.float64)
    else:
        m = z.mean(dim=(2, 3))
        h = (m @ _bf16(sd[se + "fc1.weight"].double()).reshape(128, 256).T + sd[se + "fc1.bias"].double()).clamp_min(0)
        gate = torch.sigmoid(h @ _bf16(sd[se + "fc2.weight"].double()).reshape(256, 128).T + sd[se + "fc2.bias"].double())
        gate = gate[:, :, None, None]
    return (gate * _bf16(z) + resid).clamp_min(0), z, gate, a


def _engine(blob, monkeypatch, env=None, max_batch=512):
    import scb200

    return _engine_any(blob, monkeypatch, env, max_batch, scb200.SC_MODE_FP8)


# ---- 1 / 2. every layer against float64, on all test nets -------------------------------------------------------
def _check_layers(tag, sd, stressed, e, pos, boards=None):
    """test_gpu_fp16._check_layers with e4m3 rounding: layer k from the k - 1 call's buffers.  Bound: one e4m3 ulp of
    the (saturated) reference, the fp32-accumulation floor of test_gpu_layer_reference and, for SE layers, the bf16
    park's ulp times the gate; at least BIT_EQUAL_MIN of the live elements bit-equal."""
    import net

    n = len(pos)
    boards = np.arange(n) if boards is None else np.asarray(boards)
    planes, _ = e.encode_only(pos)
    prev = [np.zeros((n, 64, 256), np.uint16) for _ in range(3)]
    prev_planes = net.planes_i8_hwc_to_nchw(planes[boards]).double()
    failures = []
    for k, layer in enumerate(_layers(sd), start=1):
        cur = e.debug_tower(pos, k, 0)
        conv, _, reads, writes, _, se = layer
        for b in (X, T, Y):
            if b != writes:
                assert np.array_equal(cur[b], prev[b]), f"{tag} layer {k} ({conv}) changed buffer {'xty'[b]}"
        inp = prev_planes if reads == PLANES else _nhwc_to_nchw(_u16_to_f64(prev[reads][boards]))
        resid = _nhwc_to_nchw(_u16_to_f64(prev[X][boards])) if se is not None else None
        ref, z, gate, a = _layer_reference(sd, layer, inp, resid)
        got = _nhwc_to_nchw(_u16_to_f64(cur[writes][boards])).numpy()
        ref = ref.clamp(-E4M3_MAX, E4M3_MAX).numpy()
        err = np.abs(got - ref)
        if layer[1] + ".weight" in sd:
            scale = np.abs(sd[layer[1] + ".weight"].double().numpy()).reshape(1, -1, 1, 1)
        else:
            scale = a.std(dim=1, unbiased=False, keepdim=True).numpy()
        g = 1.0 if gate is None else gate.numpy()
        floor = 2e-5 * scale * g + 1e-6
        if k - 1 in stressed:
            ratio = stressed[k - 1] / a.std(dim=1, unbiased=False, keepdim=True).numpy()
            shift_tol = (1e-3 + 4 * ratio * 2.0 ** -24) * scale * g
        else:
            shift_tol = 0.0
        tol = _ulp8(ref) + floor + shift_tol
        if z is not None:
            tol = tol + gate.numpy() * _ulp_bf16(z.numpy())
        want = _rnd8(torch.from_numpy(ref)).numpy()
        live = (want != 0) | (got != 0)
        equal = float((got == want)[live].mean())
        sat = float((np.abs(got) == E4M3_MAX).mean())
        print(f"{tag} n={n} layer {k:2d} {conv:22s} max err / bound {float(np.max(err / tol)):6.3f}  "
              f"bit-equal {equal:.5f} of {live.mean():.2f}  saturated {sat:.2e}")
        assert np.isfinite(got).all(), f"{tag} layer {k} ({conv}): non-finite output"
        if not (err <= tol).all():
            i = np.unravel_index(np.argmax(err - tol), err.shape)
            failures.append(f"layer {k} ({conv}): {int((err > tol).sum())} elements out of bound, worst at {i}: "
                            f"got {got[i]:.6g} ref {ref[i]:.6g}")
        if k - 1 not in stressed and equal < BIT_EQUAL_MIN:
            failures.append(f"layer {k} ({conv}): bit-equal fraction {equal:.4f} < {BIT_EQUAL_MIN}")
        prev = cur
    assert not failures, f"{tag} n={n}:\n" + "\n".join(failures)


@pytest.mark.parametrize("tag", ["n2", "stress", "bn_se", "ln_nose", "bn_nose"])
def test_fp8_tower_layers(nets, games, monkeypatch, tag):  # noqa: F811
    sd, blob, stressed = nets[tag]
    e = _engine(blob, monkeypatch)
    try:
        for n in (1, 6):
            pos, _, _ = _batch(games, n)
            _check_layers(tag, sd, stressed, e, pos)
        if tag in ("n2", "stress"):
            pos, _, _ = _batch(games, 333)
            _check_layers(tag, sd, stressed, e, pos, boards=[0, 1, 2, 3, 127, 128, 329, 330, 331, 332])
    finally:
        e.close()


def _heads_reference(sd, t, y, meta):
    lg = _conv_bias(sd, "policy_head.model.2", t)
    lg = _norm(sd, "policy_head.model.3", lg)
    logp = torch.log_softmax(lg.flatten(1), dim=1)
    w1 = sd["value_head.ffn.0.weight"].double()
    w1 = torch.cat((_scaled_weight(w1[:, :64 * 256]), w1[:, 64 * 256:]), dim=1)
    hid = (torch.cat((y.flatten(1), meta), dim=1) @ w1.T + sd["value_head.ffn.0.bias"].double()).clamp_min(0)
    v = torch.tanh(hid @ sd["value_head.ffn.2.weight"].double().T + sd["value_head.ffn.2.bias"].double())
    return logp.numpy(), (v[:, 0] * (meta[:, 0] * 2 - 1)).numpy()


@pytest.mark.parametrize("tag", ["n2", "stress", "bn_se", "ln_nose", "bn_nose"])
def test_fp8_heads_from_tower_buffers(nets, games, monkeypatch, tag):  # noqa: F811
    """the policy conv (e4m3, scaled) + LayerNorm(73) + log-softmax and the value FC (e4m3, scaled per hidden unit) +
    tail, from the tower's own e4m3 t / y buffers, against float64, at the fp16 test's tolerances"""
    import net

    sd, blob, _ = nets[tag]
    e = _engine(blob, monkeypatch)
    try:
        for n in (37, 333):
            pos, _, _ = _batch(games, n)
            planes, meta = e.encode_only(pos)
            _, t, y = e.debug_tower(pos, len(_layers(sd)), 0)
            lp, v = e.forward_only(net.planes_i8_hwc_to_nchw(planes).numpy(), meta.astype(np.float32))
            lp_ref, v_ref = _heads_reference(sd, _nhwc_to_nchw(_u16_to_f64(t)), _nhwc_to_nchw(_u16_to_f64(y)),
                                             torch.from_numpy(meta).double())
            dl, dv = float(np.abs(lp - lp_ref).max()), float(np.abs(v - v_ref).max())
            print(f"fp8 {tag} heads n={n}: max |d logp| {dl:.2e}  max |d value| {dv:.2e}")
            assert dl <= 1e-4 and dv <= 1e-5, (tag, n, dl, dv)
    finally:
        e.close()


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


@pytest.mark.parametrize("env", [{"SCB200_TOWER": "0"}, {"SCB200_TOWER_GROUP": "0"}, {"SCB200_FUSE_GATHER": "0"},
                                 {"SCB200_FUSE_VALUE": "0"}])
def test_fp8_launch_variants_bit_identical(net19, batch2048, monkeypatch, env):  # noqa: F811
    """per-layer launches, other tile groupings and the stand-alone value tail give the same bits; the stand-alone
    legal-move gather gives the same values and priors within 2e-6, as in bf16 mode"""
    import scb200

    games, pos, moves, off, mv_all, lp, v, pri_ref = batch2048
    for n in (2048, 100):
        a = _eval(net19[1], monkeypatch, pos[:n], moves[: off[n]], off[: n + 1], mode=scb200.SC_MODE_FP8)
        b = _eval(net19[1], monkeypatch, pos[:n], moves[: off[n]], off[: n + 1], env=env, mode=scb200.SC_MODE_FP8)
        assert np.array_equal(a[1], b[1]), (env, n)
        if "SCB200_FUSE_GATHER" in env:
            assert np.abs(a[0] - b[0]).max() < 2e-6, (env, n)
        else:
            assert np.array_equal(a[0], b[0]), (env, n)


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
    import scb200

    blob = nets["n2"][1]
    eng = _engine(blob, monkeypatch, max_batch=64)
    try:
        sp = scb200.SelfPlay(eng, n_trees=32, rollout_num=30, num_steps=12, cpuct=2.5, with_noise=False,
                             temperature_switch=3, temperature=0.0, keep_traces=True, pipeline_groups=2, seed=0)
        st = sp.run(max_games=32)
        assert st["games_finished"] == 32
        traces = [sp.trace(k) for k in range(32)]
        sp.close()
        for tr in traces:
            g = co.Game()
            for mv, _, ch in tr["steps"]:
                assert mv in g.legal_uci()
                g.push(mv)
        mirror = scb200.game_selfplay(eng, rollout_num=30, num_steps=12, cpuct=2.5, temperature_switch=3, seed=0)
        assert mirror == traces[0]
        eb = _engine_any(blob, monkeypatch, max_batch=64, mode=scb200.SC_MODE_BF16)
        try:
            a = scb200.Arena(eng, eb, n_trees=16, rollout=20, cpuct=1.5, temperature=0.0, temperature_switch=0,
                             max_plies=6, seed=1, keep_traces=True, n_threads=2)
            st = a.run(max_games=16)
            a.close()
            assert st["games_finished"] == 16 and st["moves"] == 16 * 6
        finally:
            eb.close()
    finally:
        eng.close()


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
