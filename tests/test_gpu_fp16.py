"""SC_MODE_FP16: the bf16 tensor-core kernels with fp16 operands.

fp16 mode rounds exactly where bf16 mode rounds, to fp16 instead of bf16 (round to nearest even): the conv, SE and
value-FC weights, each layer's stored output, the SE layers' parked z and the residual stream x.  Everything else is the
same fp32 arithmetic.  fp16 keeps 11 significant bits where bf16 keeps 8, so its error against the fp32 oracle should be
about 1/8 of bf16's; these tests hold it to at most 1/3, and check the per-layer rounding, the bit-identity of the
kernels and launch structures, the drivers and the weight range check.
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import games_to_batch
from test_gpu_bench_config import batch2048, net19  # noqa: F401  (fixtures)
from test_gpu_layer_reference import (  # noqa: F401  (fixtures and dtype-free helpers)
    LAT_SHAPES, PLANES, X, T, Y, BIT_EQUAL_MIN, _batch, _engine_tensors, _layers, _norm, _nhwc_to_nchw, games, nets)

pytestmark = pytest.mark.gpu


# ---- fp16 arithmetic of the reference ---------------------------------------------------------------------------
def _rnd16(t):
    return t.to(torch.float16).to(torch.float64)


def _u16_to_f64(u):
    return torch.from_numpy(u.view(np.float16).astype(np.float64))


def _ulp16(v):
    """Spacing of fp16 numbers at |v|: 2^(e - 11) for normal numbers, 2^-24 below 2^-14 (0 at 0)."""
    m, e = np.frexp(np.abs(v))
    return np.where(v == 0, 0.0, np.ldexp(1.0, np.maximum(e - 11, -24)))


def _conv_bias(sd, conv, x):
    w = _rnd16(sd[conv + ".weight"].double())
    return F.conv2d(x, w, sd[conv + ".bias"].double(), padding=w.shape[-1] // 2)


def _layer_reference(sd, layer, inp, resid):
    """One layer in float64 on the kernel's inputs, fp16 where the kernel rounds -> (out before the final rounding,
    z, gate, a = conv + bias).  (test_gpu_layer_reference's bf16 version with the operand type swapped.)"""
    conv, norm, _, _, relu, se = layer
    a = _conv_bias(sd, conv, inp)
    z = _norm(sd, norm, a)
    if se is None:
        return (z.clamp_min(0) if relu else z), None, None, a
    if se == "residual":
        gate = torch.ones(z.shape[0], z.shape[1], 1, 1, dtype=torch.float64)
    else:
        m = z.mean(dim=(2, 3))
        h = (m @ _rnd16(sd[se + "fc1.weight"].double()).reshape(128, 256).T + sd[se + "fc1.bias"].double()).clamp_min(0)
        gate = torch.sigmoid(h @ _rnd16(sd[se + "fc2.weight"].double()).reshape(256, 128).T + sd[se + "fc2.bias"].double())
        gate = gate[:, :, None, None]
    return (gate * _rnd16(z) + resid).clamp_min(0), z, gate, a


def forward_fp16_operands(sd, planes, meta):
    """Emulation of fp16 mode on the CPU: every conv / linear rounds its input and weight to fp16 and accumulates in
    fp32; the SE weights are fp16; everything else fp32 (the fp16 form of oracle.net.forward_bf16_operands)."""
    import net

    q = {k: (v.half().float() if v.ndim > 1 else v) for k, v in sd.items()}

    def rnd(t):
        return t.half().float()

    def conv(x, w, b, pad=0):
        return F.conv2d(rnd(x), w, b, padding=pad)

    x = conv(planes.float(), q["conv_block.0.weight"], q["conv_block.0.bias"], 1)
    x = F.relu(net.layer_norm_2d(x, q["conv_block.1.weight"], q["conv_block.1.bias"]))
    for i in range(net.n_res_blocks_of(sd)):
        p = f"res_blocks.{i}."
        o = conv(x, q[p + "conv1.weight"], q[p + "conv1.bias"], 1)
        o = F.relu(net.layer_norm_2d(o, q[p + "bn1.weight"], q[p + "bn1.bias"]))
        o = conv(o, q[p + "conv2.weight"], q[p + "conv2.bias"], 1)
        o = net.layer_norm_2d(o, q[p + "bn2.weight"], q[p + "bn2.bias"])
        s = F.adaptive_avg_pool2d(o, 1)
        s = F.relu(F.conv2d(s, q[p + "se.fc1.weight"], sd[p + "se.fc1.bias"]))
        s = torch.sigmoid(F.conv2d(s, q[p + "se.fc2.weight"], sd[p + "se.fc2.bias"]))
        x = F.relu(s * rnd(o) + x)
    ph = "policy_head.model."
    y = conv(x, q[ph + "0.weight"], q[ph + "0.bias"])
    y = net.layer_norm_2d(y, q[ph + "1.weight"], q[ph + "1.bias"])
    y = conv(y, q[ph + "2.weight"], q[ph + "2.bias"])
    y = net.layer_norm_2d(y, q[ph + "3.weight"], q[ph + "3.bias"])
    logp = F.log_softmax(y.flatten(1), dim=1)
    vh = "value_head."
    z = conv(x, q[vh + "conv.0.weight"], q[vh + "conv.0.bias"])
    z = F.relu(net.layer_norm_2d(z, q[vh + "conv.1.weight"], q[vh + "conv.1.bias"])).flatten(1)
    w1 = sd[vh + "ffn.0.weight"]
    w1 = torch.cat((w1[:, :64 * 256].half().float(), w1[:, 64 * 256:]), dim=1)
    z = F.relu(F.linear(torch.cat((rnd(z), meta.float()), dim=1), w1, sd[vh + "ffn.0.bias"]))
    v = torch.tanh(F.linear(z, sd[vh + "ffn.2.weight"], sd[vh + "ffn.2.bias"]))
    return logp, v * (meta[:, 0:1].float() * 2 - 1)


def _engine(blob, monkeypatch, env=None, max_batch=512, mode=None):
    import scb200

    for k in ("SCB200_LATENCY", "SCB200_LAT_CLUSTER", "SCB200_LAT_ONE_BOARD", "SCB200_TOWER", "SCB200_TOWER_GROUP",
              "SCB200_FUSE_GATHER", "SCB200_FUSE_VALUE"):
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    return scb200.Engine(blob, 0, scb200.SC_MODE_FP16 if mode is None else mode, max_batch)


def _eval(blob, monkeypatch, pos, moves, off, env=None, mode=None, max_batch=2048):
    e = _engine(blob, monkeypatch, env, max_batch, mode)
    try:
        pri, val = e.eval(pos, moves, off)
        return pri.copy(), val.copy()
    finally:
        e.close()


# ---- 1. the bench workload against the oracle -------------------------------------------------------------------
def test_fp16_bench_workload_vs_oracle(net19, batch2048, monkeypatch):  # noqa: F811
    """19 blocks, 2048 random-play leaves: fp16's max |d| against the fp32 oracle is at most 1/3 of bf16's on the
    same batch, for priors and values separately (expected ~1/8 from the 2^-11 / 2^-8 unit roundoffs)."""
    import scb200

    games, pos, moves, off, mv_all, lp, v, pri_ref = batch2048
    p16, v16 = _eval(net19[1], monkeypatch, pos, moves, off)
    pb, vb = _eval(net19[1], monkeypatch, pos, moves, off, mode=scb200.SC_MODE_BF16)
    assert np.isfinite(p16).all() and np.isfinite(v16).all()
    dp16, dv16 = float(np.abs(p16 - pri_ref).max()), float(np.abs(v16 - v).max())
    dpb, dvb = float(np.abs(pb - pri_ref).max()), float(np.abs(vb - v).max())
    print(f"2048 leaves vs oracle: fp16 max|d prior| {dp16:.3e} max|d value| {dv16:.3e}; "
          f"bf16 {dpb:.3e} {dvb:.3e}; ratios {dp16 / dpb:.3f} {dv16 / dvb:.3f}")
    assert dp16 <= dpb / 3 and dv16 <= dvb / 3
    agree = tot = 0
    for i in range(len(games)):
        r = pri_ref[off[i]:off[i + 1]]
        if len(r) > 1:
            s = np.sort(r)
            if s[-1] - s[-2] > 2 * dp16:
                tot += 1
                agree += int(np.argmax(p16[off[i]:off[i + 1]]) == np.argmax(r))
    print(f"top move agrees on {agree} of {tot} leaves with an oracle margin > 2 x {dp16:.2e}")
    assert agree == tot


# ---- 2. fp16-operand emulation ----------------------------------------------------------------------------------
def test_fp16_mode_deviation_is_operand_rounding(co, nets, games, monkeypatch):  # noqa: F811
    """Engine vs the CPU emulation of fp16 operands vs fp32, on the 2- and 19-block nets: the engine's deviation from
    fp32 is of the size of the operand rounding."""
    import net

    gs, depths = games
    for key, n in (("n2", 64), ("n19", 24)):
        sd = _engine_tensors(nets[key][0])
        sub, dp = gs[:n], depths[:n]
        planes = np.stack([g.encode(d)[0] for g, d in zip(sub, dp)])
        meta = np.stack([g.encode(d)[1] for g, d in zip(sub, dp)])
        x = net.planes_i8_hwc_to_nchw(planes)
        m = torch.from_numpy(meta).float()
        lp32, v32 = net.forward(sd, x, m)
        lpe, ve = forward_fp16_operands(sd, x, m)
        e = _engine(nets[key][1], monkeypatch, max_batch=64)
        try:
            lpg, vg = e.forward_only(x.numpy(), meta.astype(np.float32))
        finally:
            e.close()
        p32, pe, pg = np.exp(lp32.numpy()), np.exp(lpe.numpy()), np.exp(lpg)
        d_emu = max(np.abs(pg - pe).max(), np.abs(vg - ve.numpy().reshape(-1)).max())
        d_f32 = max(np.abs(pg - p32).max(), np.abs(vg - v32.numpy().reshape(-1)).max())
        d_ref = max(np.abs(pe - p32).max(), np.abs(ve.numpy() - v32.numpy()).max())
        print(f"{key}: |gpu - fp16 emulation| {d_emu:.2e}  |gpu - fp32| {d_f32:.2e}  |emulation - fp32| {d_ref:.2e}")
        assert d_f32 < 4 * d_ref + 1e-4


# ---- 3. every layer against float64 -----------------------------------------------------------------------------
def _check_layers(tag, sd, stressed, e, pos, which, boards=None):
    """test_gpu_layer_reference._check_layers with fp16 rounding: layer k from the k - 1 call's buffers."""
    import net

    n = len(pos)
    boards = np.arange(n) if boards is None else np.asarray(boards)
    planes, _ = e.encode_only(pos)
    prev = [np.zeros((n, 64, 256), np.uint16) for _ in range(3)]
    prev_planes = net.planes_i8_hwc_to_nchw(planes[boards]).double()
    failures = []
    for k, layer in enumerate(_layers(sd), start=1):
        cur = e.debug_tower(pos, k, which)
        conv, _, reads, writes, _, se = layer
        for b in (X, T, Y):
            if b != writes:
                assert np.array_equal(cur[b], prev[b]), f"{tag} which={which} layer {k} ({conv}) changed buffer {'xty'[b]}"
        inp = prev_planes if reads == PLANES else _nhwc_to_nchw(_u16_to_f64(prev[reads][boards]))
        resid = _nhwc_to_nchw(_u16_to_f64(prev[X][boards])) if se is not None else None
        ref, z, gate, a = _layer_reference(sd, layer, inp, resid)
        got = _nhwc_to_nchw(_u16_to_f64(cur[writes][boards])).numpy()
        ref = ref.numpy()
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
        tol = _ulp16(ref) + floor + shift_tol
        if z is not None:
            tol = tol + gate.numpy() * _ulp16(z.numpy())
        want = _rnd16(torch.from_numpy(ref)).numpy()
        live = (want != 0) | (got != 0)
        equal = float((got == want)[live].mean())
        print(f"{tag} which={which} n={n} layer {k:2d} {conv:22s} max err / bound {float(np.max(err / tol)):6.3f}  "
              f"bit-equal {equal:.5f} of {live.mean():.2f}")
        assert np.isfinite(got).all(), f"{tag} layer {k} ({conv}): non-finite output"
        if not (err <= tol).all():
            i = np.unravel_index(np.argmax(err - tol), err.shape)
            failures.append(f"layer {k} ({conv}): {int((err > tol).sum())} elements out of bound, worst at {i}: "
                            f"got {got[i]:.6g} ref {ref[i]:.6g}")
        if k - 1 not in stressed and equal < BIT_EQUAL_MIN:
            failures.append(f"layer {k} ({conv}): bit-equal fraction {equal:.4f} < {BIT_EQUAL_MIN}")
        prev = cur
    assert not failures, f"{tag} which={which} n={n}:\n" + "\n".join(failures)


@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_fp16_throughput_kernel_layers(nets, games, monkeypatch, tag):  # noqa: F811
    sd, blob, stressed = nets[tag]
    e = _engine(blob, monkeypatch)
    try:
        for n in (1, 3, 6):
            pos, _, _ = _batch(games, n)
            _check_layers(tag, sd, stressed, e, pos, 0)
        pos, _, _ = _batch(games, 333)
        _check_layers(tag, sd, stressed, e, pos, 0, boards=[0, 1, 2, 3, 127, 128, 329, 330, 331, 332])
    finally:
        e.close()


@pytest.mark.parametrize("shape", sorted(LAT_SHAPES))
@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_fp16_latency_kernel_layers(nets, games, monkeypatch, tag, shape):  # noqa: F811
    sd, blob, stressed = nets[tag]
    e = _engine(blob, monkeypatch, LAT_SHAPES[shape], max_batch=16)
    try:
        for n in (1, 5):
            pos, _, _ = _batch(games, n)
            _check_layers(f"{tag}/{shape}", sd, stressed, e, pos, 1)
    finally:
        e.close()


def _heads_reference(sd, t, y, meta):
    lg = _conv_bias(sd, "policy_head.model.2", t)
    lg = _norm(sd, "policy_head.model.3", lg)
    logp = torch.log_softmax(lg.flatten(1), dim=1)
    w1 = sd["value_head.ffn.0.weight"].double()
    w1 = torch.cat((_rnd16(w1[:, :64 * 256]), w1[:, 64 * 256:]), dim=1)
    hid = (torch.cat((y.flatten(1), meta), dim=1) @ w1.T + sd["value_head.ffn.0.bias"].double()).clamp_min(0)
    v = torch.tanh(hid @ sd["value_head.ffn.2.weight"].double().T + sd["value_head.ffn.2.bias"].double())
    return logp.numpy(), (v[:, 0] * (meta[:, 0] * 2 - 1)).numpy()


@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_fp16_heads_from_tower_buffers(nets, games, monkeypatch, tag):  # noqa: F811
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
            print(f"fp16 {tag} heads n={n}: max |d logp| {dl:.2e}  max |d value| {dv:.2e}")
            assert dl <= 1e-4 and dv <= 1e-5, (tag, n, dl, dv)
    finally:
        e.close()


# ---- 4. latency kernel == throughput kernel ---------------------------------------------------------------------
LAT_SIZES = (1, 2, 3, 7, 16, 33, 36, 37, 64, 74, 75, 96)


@pytest.mark.parametrize("env", [{}, {"SCB200_LAT_CLUSTER": "4"}, {"SCB200_LAT_CLUSTER": "8"},
                                 {"SCB200_LAT_ONE_BOARD": "0"}])
def test_fp16_latency_equals_throughput(nets, games, monkeypatch, env):  # noqa: F811
    blob = nets["n2"][1]
    pos, moves, off = _batch(games, 96)
    ref = _engine(blob, monkeypatch, {"SCB200_LATENCY": "0"}, max_batch=96)
    lat = _engine(blob, monkeypatch, env, max_batch=96)
    try:
        for n in LAT_SIZES:
            a = ref.eval(pos[:n], moves[: off[n]], off[: n + 1])
            b = lat.eval(pos[:n], moves[: off[n]], off[: n + 1])
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), (env, n)
        full = lat.eval(pos, moves, off)
        full = (full[0].copy(), full[1].copy())
        for i in (0, 17, 95):
            o = off[i:i + 2] - off[i]
            p1, v1 = lat.eval(pos[i:i + 1], moves[off[i]:off[i + 1]], o)
            assert np.array_equal(p1, full[0][off[i]:off[i + 1]]) and v1[0] == full[1][i]
    finally:
        ref.close()
        lat.close()


# ---- 5. launch structures and fused paths -----------------------------------------------------------------------
@pytest.mark.parametrize("env", [{"SCB200_TOWER": "0"}, {"SCB200_TOWER_GROUP": "0"}, {"SCB200_FUSE_GATHER": "0"},
                                 {"SCB200_FUSE_VALUE": "0"}])
def test_fp16_launch_variants_bit_identical(net19, batch2048, monkeypatch, env):  # noqa: F811
    """Per-layer launches, other tile groupings and the stand-alone value tail give the same bits as the defaults.  The
    stand-alone legal-move gather (policy.cu) is the fused epilogue's arithmetic in another kernel, not the same
    instruction sequence: as in bf16 mode (test_fused_policy_gather_matches_standalone_kernel) the values are bit-equal
    and the priors agree to 2e-6."""
    games, pos, moves, off, mv_all, lp, v, pri_ref = batch2048
    for n in (2048, 100):
        a = _eval(net19[1], monkeypatch, pos[:n], moves[: off[n]], off[: n + 1], env={"SCB200_LATENCY": "0"})
        b = _eval(net19[1], monkeypatch, pos[:n], moves[: off[n]], off[: n + 1], env=dict(env, SCB200_LATENCY="0"))
        assert np.array_equal(a[1], b[1]), (env, n)
        if "SCB200_FUSE_GATHER" in env:
            assert np.abs(a[0] - b[0]).max() < 2e-6, (env, n)
        else:
            assert np.array_equal(a[0], b[0]), (env, n)


# ---- 6. network variants ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("tag", ["bn_se", "ln_nose", "bn_nose"])
def test_fp16_variant_networks(co, net_golden, tmp_path, tag, monkeypatch):
    """BatchNorm (folded) and residual-only variants against the oracle and the module.py goldens, at 1/3 of the 2e-2
    tolerance bf16 passes them at."""
    import net
    import scb200

    tol = 2e-2 / 3
    info = net_golden["info"]["variants"][tag]
    sd = net.init_variant_state_dict(info["n_res_blocks"], info["seed"], info["norm"], info["use_se"])
    blob = str(tmp_path / f"{tag}.scw")
    scb200.write_blob(sd, blob)
    gs = co.random_play_positions(70, seed=41)
    pos, moves, off, mv_all = games_to_batch(gs)
    planes = np.stack([g.encode()[0] for g in gs])
    meta = np.stack([g.encode()[1] for g in gs])
    x = net.planes_i8_hwc_to_nchw(planes)
    lp, v = net.forward(sd, x, torch.from_numpy(meta).float())
    lp, v = lp.numpy(), v.numpy().reshape(-1)
    ref = np.concatenate([co.post_process(lp[i], g.move_indices(mv)) for i, (g, mv) in enumerate(zip(gs, mv_all))])
    xg = net.planes_i8_hwc_to_nchw(net_golden["planes_i8"]).numpy()
    mg = net_golden["meta_i32"].astype(np.float32)
    same_net = abs(net.state_dict_digest({k: t for k, t in sd.items() if t.ndim > 0})["sum"] - info["digest"]["sum"]) < 1e-6
    e = _engine(blob, monkeypatch, max_batch=128)
    try:
        lp_g, v_g = e.forward_only(x.numpy(), meta.astype(np.float32))
        pri, val = e.eval(pos, moves, off)
        d = (np.abs(np.exp(lp_g) - np.exp(lp)).max(), np.abs(v_g - v).max(), np.abs(pri - ref).max(),
             np.abs(val - v).max())
        print(tag, "fp16 max diffs (p, value, prior, value)", ["%.2e" % t for t in d])
        assert max(d) < tol
        if same_net:
            lg, vg = e.forward_only(xg, mg)
            assert np.abs(np.exp(lg) - np.exp(net_golden["logp_" + tag])).max() < tol
            assert np.abs(vg - net_golden["value_" + tag]).max() < tol
    finally:
        e.close()


# ---- 7. drivers -------------------------------------------------------------------------------------------------
def test_fp16_selfplay_arena_and_game(co, nets, monkeypatch, tmp_path):  # noqa: F811
    import scb200

    blob = nets["n2"][1]
    eng = _engine(blob, monkeypatch, max_batch=64)
    try:
        runs = []
        for _ in range(2):
            sp = scb200.SelfPlay(eng, n_trees=32, rollout_num=30, num_steps=12, cpuct=2.5, with_noise=False,
                                 temperature_switch=3, temperature=0.0, keep_traces=True, pipeline_groups=2, seed=0)
            st = sp.run(max_games=32)
            assert st["games_finished"] == 32
            runs.append([sp.trace(k) for k in range(32)])
            sp.close()
        assert runs[0] == runs[1]
        for tr in runs[0]:
            g = co.Game()
            for mv, _, ch in tr["steps"]:
                assert mv in g.legal_uci()
                g.push(mv)
        mirror = scb200.game_selfplay(eng, rollout_num=30, num_steps=12, cpuct=2.5, temperature_switch=3, seed=0)
        assert mirror == runs[0][0]
        eb = _engine(blob, monkeypatch, max_batch=64, mode=scb200.SC_MODE_BF16)
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


def test_fp16_golden_game_first_divergence(tmp_path):
    """Printed, not gated: the first ply at which fp16 / bf16 leave the configs[0] golden visit tables (fp32 replays
    all of them)."""
    import scb200

    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "search_cfg1.json")))
    cfg = gold["config"]
    blob = str(tmp_path / "seed0.scw")
    scb200.write_blob(scb200.random_init_state_dict(cfg["n_res_blocks"], 0), blob)
    for name, mode in (("fp16", scb200.SC_MODE_FP16), ("bf16", scb200.SC_MODE_BF16)):
        eng = scb200.Engine(blob, 0, mode, 4)
        sp = scb200.SelfPlay(eng, n_trees=2, rollout_num=cfg["rollout_num"], num_steps=cfg["num_steps"],
                             cpuct=cfg["cpuct"], with_noise=False, temperature_switch=0, temperature=0.0,
                             keep_traces=True, pipeline_groups=2)
        sp.run(max_games=2)
        tr = sp.trace(0)
        sp.close()
        eng.close()
        first = None
        for ply, ((mv, q, ch), ref) in enumerate(zip(tr["steps"], gold["steps"])):
            if mv != ref["move"] or [c[1] for c in ch] != [c[1] for c in ref["children"]]:
                first = ply
                break
        print(f"{name}: first ply off the configs[0] golden visit tables: {first} (golden plies {len(gold['steps'])})")


# ---- 8. weight range check --------------------------------------------------------------------------------------
def test_fp16_rejects_weights_beyond_range(nets, tmp_path):  # noqa: F811
    import net
    import scb200

    sd = net.init_state_dict(2, 7)
    sd["res_blocks.1.conv1.weight"].view(-1)[123] = 1e5
    blob = str(tmp_path / "big.scw")
    scb200.write_blob(sd, blob)
    with pytest.raises(scb200.SCError) as ei:
        scb200.Engine(blob, 0, scb200.SC_MODE_FP16, 4)
    msg = str(ei.value)
    print(msg)
    assert "(-3)" in msg and "res_blocks.1.conv1.weight" in msg and "65504" in msg      # SC_E_IO, naming the tensor
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 4)       # bf16 has the fp32 exponent range
    e.close()
