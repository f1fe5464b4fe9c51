"""SC_MODE_FP16: the bf16 tensor-core kernels with fp16 operands.

fp16 mode rounds exactly where bf16 mode rounds, to fp16 instead of bf16 (round to nearest even): the conv, SE and
value-FC weights, each layer's stored output, the SE layers' parked z and the residual stream x.  Everything else is the
same fp32 arithmetic.  fp16 keeps 11 significant bits where bf16 keeps 8, so its error against the fp32 oracle should be
about 1/8 of bf16's; these tests hold it to at most 1/3, and check the bit-identity of the latency and throughput kernels,
the per-layer rounding, the launch structures, the network variants, the drivers and the weight range check.  The
per-layer and heads references and the launch-variant and driver checks are test_gpu_layer_reference's, shared with
the other tensor-core modes.
"""
import functools
import json
import os

import numpy as np
import pytest
import scb200
import torch
import torch.nn.functional as F

from conftest import games_to_batch
from test_gpu_bench_config import batch2048, net19  # noqa: F401  (fixtures)
from test_gpu_layer_reference import (  # noqa: F401  (fixtures)
    FP16, LAT_SHAPES, LAUNCH_VARIANTS, _batch, _engine as _engine_any, _engine_tensors, _eval as _eval_any,
    check_launch_variant, check_selfplay_arena_and_game, games, nets, run_heads, run_latency_layers,
    run_throughput_layers)

pytestmark = pytest.mark.gpu

_engine = functools.partial(_engine_any, mode=scb200.SC_MODE_FP16)
_eval = functools.partial(_eval_any, mode=scb200.SC_MODE_FP16)


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
@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_fp16_throughput_kernel_layers(nets, games, monkeypatch, tag):  # noqa: F811
    run_throughput_layers(FP16, nets, games, monkeypatch, tag, (1, 3, 6), [0, 1, 2, 3, 127, 128, 329, 330, 331, 332])


@pytest.mark.parametrize("shape", sorted(LAT_SHAPES))
@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_fp16_latency_kernel_layers(nets, games, monkeypatch, tag, shape):  # noqa: F811
    run_latency_layers(FP16, nets, games, monkeypatch, tag, shape)


@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_fp16_heads_from_tower_buffers(nets, games, monkeypatch, tag):  # noqa: F811
    run_heads(FP16, nets, games, monkeypatch, tag)


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
@pytest.mark.parametrize("env", LAUNCH_VARIANTS)
def test_fp16_launch_variants_bit_identical(net19, batch2048, monkeypatch, env):  # noqa: F811
    check_launch_variant(scb200.SC_MODE_FP16, net19, batch2048, monkeypatch, env)


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
    check_selfplay_arena_and_game(scb200.SC_MODE_FP16, co, nets, monkeypatch)


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
