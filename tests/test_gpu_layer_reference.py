"""Every layer of the tensor-core tower kernels against a float64 reference of the same layer (sc_debug_tower), for
each operand type: bf16, fp16 and e4m3 (SC_MODE_BF16 / SC_MODE_FP16 / SC_MODE_FP8).

The end-to-end bf16 checks compare with the fp32 oracle at 2e-2, and every layer renormalises its output, so a small
arithmetic error in an epilogue (a pooling divisor, a rounding mode, a dropped term) is damped layer after layer and
hides inside that tolerance.  The latency and throughput kernels share their LayerNorm and SE arithmetic, so the
bit-identity tests between them cannot see an error in it either.  Here each layer's output is compared with a float64
computation of that one layer on the kernel's own inputs, rounded only where the kernel documents a rounding (`Format`
below holds the roundings of each operand type):

  * convolution weights as `load_weights` packs them (bf16 / fp16; e4m3 with a power-of-two scale per output channel),
    SE weights in the type the SE layers park values in (bf16 for bf16 and e4m3, fp16 for fp16), bias / gamma / beta
    in fp32;
  * conv + bias and the LayerNorm in float64 (folded-BatchNorm nets have no normalisation);
  * LayerNorm layers: one rounding to the operand type at the output (e4m3 saturates at +-448);
  * LayerNorm + SE layers: pool the unrounded z = LN(conv + b), gate g = sigmoid(W2 relu(W1 mean + b1) + b2)
    (g = 1 for residual-only blocks), out = rnd(relu(g * park(z) + x)).

Per layer every element must be within one ulp of the (for e4m3 saturated) reference (plus g ulps of the parked z,
plus a small allowance for the fp32 accumulation of the convolution), at least 99 % of the elements that are non-zero on
either side must be bit-equal to the rounded reference, and the buffers the layer does not write must be unchanged.
The head GEMMs are then checked from the tower's final t / y buffers against forward_only at the fp32 tolerances,
since their operands are the same numbers.
"""
from typing import Callable, NamedTuple, Optional

import numpy as np
import pytest
import scb200
import torch
import torch.nn.functional as F

from conftest import games_to_batch

pytestmark = pytest.mark.gpu

LN_EPS = 1e-6
BIT_EQUAL_MIN = 0.99
X, T, Y = 0, 1, 2            # sc_debug_tower buffers
PLANES = -1


# ---- weights --------------------------------------------------------------------------------------------------
def _stress_state_dict():
    """2-block LN+SE net with negative gammas, large betas and SE gates saturated toward 0 and 1 in some channels."""
    import net

    sd = net.init_variant_state_dict(2, 91, "LayerNorm", True)
    g = torch.Generator().manual_seed(92)
    for k in list(sd):
        v = sd[k]
        if v.ndim == 1 and (".bn" in k or "conv_block.1" in k or "conv.1." in k or "model.1." in k or "model.3." in k):
            if k.endswith(".weight"):
                sd[k] = 1.5 * (2 * torch.rand(v.shape, generator=g) - 1)          # some negative, some near zero
            else:
                sd[k] = 2.5 * (2 * torch.rand(v.shape, generator=g) - 1)
    for i in range(2):
        b = sd[f"res_blocks.{i}.se.fc2.bias"]
        b[0::16] = -30.0                                                           # gate -> 0
        b[5::16] = 30.0                                                            # gate -> 1
    return sd


# layers that get a common offset on every channel's conv bias, and the offset in units of the median over squares of
# the std over channels of that layer's conv + bias
STRESS_OFFSETS = {"res_blocks.0.conv1": 300.0, "res_blocks.1.conv2": 5000.0}


def _layers(sd):
    """The tower's layers in sc_debug_tower order (engine.cu): (conv, norm, reads, writes, relu, SE kind)."""
    import net

    nb = net.n_res_blocks_of(sd)
    use_se = "res_blocks.0.se.fc1.weight" in sd
    out = [("conv_block.0", "conv_block.1", PLANES, X, True, None)]
    for i in range(nb):
        p = f"res_blocks.{i}."
        out.append((p + "conv1", p + "bn1", X, T, True, None))
        out.append((p + "conv2", p + "bn2", T, X, True, p + "se." if use_se else "residual"))
    out.append(("policy_head.model.0", "policy_head.model.1", X, T, False, None))
    out.append(("value_head.conv.0", "value_head.conv.1", X, Y, True, None))
    return out


def _engine_tensors(sd):
    """The tensors the engine loads: BatchNorm folded into the convolutions exactly as scb200.export does."""
    import net
    from scb200.export import _fold_batchnorm

    if any(k.endswith("running_mean") for k in sd):
        return _fold_batchnorm(sd, net.n_res_blocks_of(sd))
    return dict(sd)


# ---- operand types ----------------------------------------------------------------------------------------------
E4M3_MAX = 448.0


def _bf16(t):
    return t.to(torch.bfloat16).to(torch.float64)


def _rnd16(t):
    return t.to(torch.float16).to(torch.float64)


def _rnd8(t):
    """round to e4m3 (nearest even), saturating at +-448 (cvt.rn.satfinite)"""
    return t.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).to(torch.float64)


def _ulp_bf16(v):
    """Spacing of bf16 numbers at |v| (0 at 0)."""
    m, e = np.frexp(np.abs(v))
    return np.where(v == 0, 0.0, np.ldexp(1.0, e - 8))


def _ulp16(v):
    """Spacing of fp16 numbers at |v|: 2^(e - 11) for normal numbers, 2^-24 below 2^-14 (0 at 0)."""
    m, e = np.frexp(np.abs(v))
    return np.where(v == 0, 0.0, np.ldexp(1.0, np.maximum(e - 11, -24)))


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


def _bf16_bits_to_f64(u):
    return torch.from_numpy((u.astype(np.uint32) << 16).view(np.float32)).double()


def _fp16_bits_to_f64(u):
    return torch.from_numpy(u.view(np.float16).astype(np.float64))


class Format(NamedTuple):
    """One tensor-core operand type as the engine uses it (tc_ptx.cuh's OpBf16 / OpFp16 / OpE4m3)."""
    name: str
    mode: int                 # SC_MODE_*
    weight: Callable          # [cout, ...] fp32 weights -> float64, as load_weights packs them
    rnd: Callable             # float64 -> the stored-output type, float64
    ulp: Callable             # numpy: the stored-output type's spacing at |v|
    park_rnd: Callable        # the SE layers' parked z and the SE weights
    park_ulp: Callable
    decode: Callable          # sc_debug_tower's uint16 buffers -> float64 (e4m3 arrives as fp16 bit patterns)
    clamp: Optional[float]    # the reference is saturated to +-clamp before the error is taken


BF16 = Format("bf16", scb200.SC_MODE_BF16, lambda w: _bf16(w.double()), _bf16, _ulp_bf16, _bf16, _ulp_bf16,
              _bf16_bits_to_f64, None)
FP16 = Format("fp16", scb200.SC_MODE_FP16, lambda w: _rnd16(w.double()), _rnd16, _ulp16, _rnd16, _ulp16,
              _fp16_bits_to_f64, None)
FP8 = Format("fp8", scb200.SC_MODE_FP8, _scaled_weight, _rnd8, _ulp8, _bf16, _ulp_bf16, _fp16_bits_to_f64, E4M3_MAX)


# ---- float64 reference ------------------------------------------------------------------------------------------
def _nhwc_to_nchw(a):             # [n, 64, C] -> [n, C, 8, 8]
    return a.reshape(a.shape[0], 8, 8, -1).permute(0, 3, 1, 2)


def _conv_bias(fmt, sd, conv, x):
    w = fmt.weight(sd[conv + ".weight"])
    return F.conv2d(x, w, sd[conv + ".bias"].double(), padding=w.shape[-1] // 2)


def _norm(sd, norm, a):
    if norm + ".weight" not in sd:                                   # folded BatchNorm: no normalisation
        return a
    mean = a.mean(dim=1, keepdim=True)
    var = ((a - mean) ** 2).mean(dim=1, keepdim=True)
    g, b = sd[norm + ".weight"].double().view(1, -1, 1, 1), sd[norm + ".bias"].double().view(1, -1, 1, 1)
    return (a - mean) / torch.sqrt(var + LN_EPS) * g + b


def _layer_reference(fmt, sd, layer, inp, resid):
    """One layer in float64 on NCHW inputs -> (out before the final rounding, z, gate, a = conv + bias)."""
    conv, norm, _, _, relu, se = layer
    a = _conv_bias(fmt, sd, conv, inp)
    z = _norm(sd, norm, a)
    if se is None:
        return (z.clamp_min(0) if relu else z), None, None, a
    if se == "residual":
        gate = torch.ones(z.shape[0], z.shape[1], 1, 1, dtype=torch.float64)
    else:
        m = z.mean(dim=(2, 3))
        w1, w2 = fmt.park_rnd(sd[se + "fc1.weight"].double()), fmt.park_rnd(sd[se + "fc2.weight"].double())
        h = (m @ w1.reshape(128, 256).T + sd[se + "fc1.bias"].double()).clamp_min(0)
        gate = torch.sigmoid(h @ w2.reshape(256, 128).T + sd[se + "fc2.bias"].double())
        gate = gate[:, :, None, None]
    return (gate * fmt.park_rnd(z) + resid).clamp_min(0), z, gate, a


def _reference_tower(fmt, sd, planes_nchw):
    """The whole tower in float64 with the kernel's hand-over between layers: per layer a = conv + bias."""
    bufs = {PLANES: planes_nchw}
    out = []
    for layer in _layers(sd):
        o, _, _, a = _layer_reference(fmt, sd, layer, bufs[layer[2]], bufs.get(X))
        bufs[layer[3]] = fmt.rnd(o)
        out.append(a)
    return out


# ---- fixtures ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def games(co, sample_games):
    """Random play plus sample-game positions cut at partial history depths (history and repetition planes set)."""
    rng = np.random.RandomState(12)
    gs, depths = [], []
    for game in sample_games["games"][:8]:
        g = co.Game()
        for u in game["uci"].split():
            g.push(u)
            if rng.rand() < 0.15 and len(g.legal_moves()) > 0:
                gs.append(g.dup())
                depths.append(int(rng.randint(0, g.ply + 1)))
    for g in co.random_play_positions(400, seed=17):
        if len(g.legal_moves()) > 0:
            gs.append(g)
            depths.append(g.ply if rng.rand() < 0.5 else int(rng.randint(0, g.ply + 1)))
    order = rng.permutation(len(gs))
    return [gs[i] for i in order], [depths[i] for i in order]


def _batch(games, n):
    gs, depths = games
    assert len(gs) >= n
    pos, moves, off, _ = games_to_batch(gs[:n], depths[:n])
    return pos, moves, off


@pytest.fixture(scope="module")
def nets(tmp_path_factory, games, net_golden):
    """name -> (the tensors the engine loads, blob path, {layer index: bias offset} of the stressed layers)."""
    import net

    d = tmp_path_factory.mktemp("layer_ref")
    sds = {"n2": net.perturb_norm_params(net.init_state_dict(2, 7), 1234), "n19": net.init_state_dict(19, 0)}
    for tag in ("bn_se", "ln_nose", "bn_nose"):
        info = net_golden["info"]["variants"][tag]
        sds[tag] = net.init_variant_state_dict(info["n_res_blocks"], info["seed"], info["norm"], info["use_se"])
    # stress: measure each stressed layer's per-square std of conv + bias on the CPU, then shift its bias by a multiple
    sd = _stress_state_dict()
    planes = np.stack([g.encode(dp)[0] for g, dp in zip(games[0][:64], games[1][:64])])
    acts = _reference_tower(BF16, sd, net.planes_i8_hwc_to_nchw(planes).double())
    names = [layer[0] for layer in _layers(sd)]
    stressed = {}
    for conv, ratio in STRESS_OFFSETS.items():
        k = names.index(conv)
        std = float(acts[k].std(dim=1, unbiased=False).median())
        sd[conv + ".bias"] = sd[conv + ".bias"] + ratio * std
        stressed[k] = ratio * std
    sds["stress"] = sd
    out = {}
    for name, s in sds.items():
        p = str(d / f"{name}.scw")
        scb200.write_blob(s, p)
        out[name] = (_engine_tensors(s), p, stressed if name == "stress" else {})
    return out


def _engine(blob, monkeypatch, env=None, max_batch=512, mode=scb200.SC_MODE_BF16):
    for k in ("SCB200_LATENCY", "SCB200_LAT_CLUSTER", "SCB200_LAT_ONE_BOARD", "SCB200_TOWER", "SCB200_TOWER_GROUP",
              "SCB200_FUSE_GATHER", "SCB200_FUSE_VALUE"):
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    return scb200.Engine(blob, 0, mode, max_batch)   # switches: read at creation


def _eval(blob, monkeypatch, pos, moves, off, env=None, mode=scb200.SC_MODE_BF16, max_batch=2048):
    e = _engine(blob, monkeypatch, env, max_batch, mode)
    try:
        pri, val = e.eval(pos, moves, off)
        return pri.copy(), val.copy()
    finally:
        e.close()


# ---- the per-layer check ----------------------------------------------------------------------------------------
def _check_layers(fmt, tag, sd, stressed, e, pos, which, boards=None):
    """Runs k = 1 .. L layers of kernel `which` and checks layer k from the k - 1 call's buffers."""
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
                assert np.array_equal(cur[b], prev[b]), \
                    f"{fmt.name} {tag} which={which} layer {k} ({conv}) changed buffer {'xty'[b]}"
        inp = prev_planes if reads == PLANES else _nhwc_to_nchw(fmt.decode(prev[reads][boards]))
        resid = _nhwc_to_nchw(fmt.decode(prev[X][boards])) if se is not None else None
        ref, z, gate, a = _layer_reference(fmt, sd, layer, inp, resid)
        got = _nhwc_to_nchw(fmt.decode(cur[writes][boards])).numpy()
        if fmt.clamp is not None:
            ref = ref.clamp(-fmt.clamp, fmt.clamp)
        ref = ref.numpy()
        err = np.abs(got - ref)
        # the fp32 accumulation of the convolution differs from float64 by about 1e-6 of the square's spread; in the
        # output that is 1e-6 |gamma| (1e-6 of the spread of z where there is no normalisation), allowed here 20 times
        if layer[1] + ".weight" in sd:
            scale = np.abs(sd[layer[1] + ".weight"].double().numpy()).reshape(1, -1, 1, 1)
        else:
            scale = a.std(dim=1, unbiased=False, keepdim=True).numpy()
        g = 1.0 if gate is None else gate.numpy()
        floor = 2e-5 * scale * g + 1e-6
        if k - 1 in stressed:
            # a = acc + bias rounded to fp32 at |a| ~ ratio x the square's spread is off by up to ratio * 2^-24 of the
            # spread in every fp32 kernel; the mean adds about twice that (the chunk sum 32 a[0] + sum d and the three
            # pairwise additions round at up to 32, 64, 128, 256 x |a|, i.e. (1/8 + 1/4 + 1/2 + 1) ratio * 2^-24
            # after the division by 256) and its own rounding once more: 4 ratio * 2^-24 in all.  ratio is the
            # square's own (offset / its spread), since a square with a smaller spread has a larger error.  On top,
            # 1e-3 of the normalised value covers the error of rstd.  No bit-equality here.
            ratio = stressed[k - 1] / a.std(dim=1, unbiased=False, keepdim=True).numpy()
            shift_tol = (1e-3 + 4 * ratio * 2.0 ** -24) * scale * g
        else:
            shift_tol = 0.0
        tol = fmt.ulp(ref) + floor + shift_tol
        if z is not None:
            tol = tol + gate.numpy() * fmt.park_ulp(z.numpy())
        # bit-equality counted where either side is non-zero: after a ReLU about half the outputs are 0 on both
        # sides, which would make the 99 % gate about 98 % on the values that carry information
        want = fmt.rnd(torch.from_numpy(ref)).numpy()
        live = (want != 0) | (got != 0)
        equal = float((got == want)[live].mean())
        worst = float(np.max(err / np.maximum(fmt.ulp(ref), 1e-6)))     # ulps, at least 1e-6
        msg = (f"{fmt.name} {tag} which={which} n={n} layer {k:2d} {conv:22s} max err {worst:8.3g} ulp  "
               f"max err / bound {float(np.max(err / tol)):6.3f}  bit-equal {equal:.5f} of {live.mean():.2f}")
        if fmt.clamp is not None:
            msg += f"  saturated {float((np.abs(got) == fmt.clamp).mean()):.2e}"
        if k - 1 in stressed:
            # the error beyond the ulp terms, as a fraction of |gamma| g: what the 1e-3 + 4 ratio 2^-24 bound is on
            excess = np.maximum(err - (tol - shift_tol), 0) / (scale * g)
            msg += f"  (shifted bias: excess {float(excess.max()):.2e} |gamma| g, ratio up to {float(ratio.max()):.0f})"
        print(msg)
        assert np.isfinite(got).all(), f"{tag} layer {k} ({conv}): non-finite output"
        if not (err <= tol).all():
            i = np.unravel_index(np.argmax(err - tol), err.shape)
            failures.append(f"layer {k} ({conv}): {int((err > tol).sum())} elements out of bound, worst at {i}: "
                            f"got {got[i]:.6g} ref {ref[i]:.6g}")
        if k - 1 not in stressed and equal < BIT_EQUAL_MIN:
            failures.append(f"layer {k} ({conv}): bit-equal fraction {equal:.4f} < {BIT_EQUAL_MIN}")
        prev = cur
    assert not failures, f"{fmt.name} {tag} which={which} n={n}:\n" + "\n".join(failures)


def run_throughput_layers(fmt, nets, games, monkeypatch, tag, sizes, boards=None):
    """The throughput kernel's layers on net `tag`: every board of a batch of each size in `sizes`, then `boards` of a
    333-board batch (several tile groups ending in a partial tile) unless None."""
    sd, blob, stressed = nets[tag]
    e = _engine(blob, monkeypatch, mode=fmt.mode)
    try:
        for n in sizes:
            pos, _, _ = _batch(games, n)
            _check_layers(fmt, tag, sd, stressed, e, pos, 0)
        if boards is not None:
            pos, _, _ = _batch(games, 333)
            _check_layers(fmt, tag, sd, stressed, e, pos, 0, boards=boards)
    finally:
        e.close()


@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_throughput_kernel_layers(nets, games, monkeypatch, tag):
    """Partial CTA-pair tiles (a pair is 4 boards) and a batch over several tile groups ending in a partial tile."""
    run_throughput_layers(BF16, nets, games, monkeypatch, tag, (1, 2, 3, 5, 6),
                          [0, 1, 2, 3, 4, 5, 127, 128, 200, 329, 330, 331, 332])


LAT_SHAPES = {"cl8_one": {"SCB200_LAT_CLUSTER": "8"}, "cl4_one": {"SCB200_LAT_CLUSTER": "4"},
              "cl8_two": {"SCB200_LAT_CLUSTER": "8", "SCB200_LAT_ONE_BOARD": "0"},
              "cl4_two": {"SCB200_LAT_CLUSTER": "4", "SCB200_LAT_ONE_BOARD": "0"}}


def run_latency_layers(fmt, nets, games, monkeypatch, tag, shape):
    """The latency kernel's layers on net `tag` in one of its shapes (LAT_SHAPES), at n = 1 and 5."""
    sd, blob, stressed = nets[tag]
    e = _engine(blob, monkeypatch, LAT_SHAPES[shape], max_batch=16, mode=fmt.mode)
    try:
        for n in (1, 5):
            pos, _, _ = _batch(games, n)
            _check_layers(fmt, f"{tag}/{shape}", sd, stressed, e, pos, 1)
    finally:
        e.close()


@pytest.mark.parametrize("shape", sorted(LAT_SHAPES))
@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_latency_kernel_layers(nets, games, monkeypatch, tag, shape):
    """Each of the latency kernel's four shapes: clusters of 8 / 4 CTAs, one- / two-board tiles."""
    run_latency_layers(BF16, nets, games, monkeypatch, tag, shape)


@pytest.mark.parametrize("tag", ["n19", "bn_se", "ln_nose", "bn_nose"])
def test_layers_other_nets(nets, games, monkeypatch, tag):
    """All 41 layers of the 19-block seed-0 net, and the folded-BatchNorm / residual-only variants, in both kernels."""
    sd, blob, stressed = nets[tag]
    e = _engine(blob, monkeypatch, max_batch=16)
    try:
        pos, _, _ = _batch(games, 3)
        for which in (0, 1):
            _check_layers(BF16, tag, sd, stressed, e, pos, which)
    finally:
        e.close()


# ---- heads ------------------------------------------------------------------------------------------------------
def _heads_reference(fmt, sd, t, y, meta):
    """Policy log-probs and value in float64 from the head GEMMs' inputs t, y (NCHW)."""
    lg = _conv_bias(fmt, sd, "policy_head.model.2", t)
    lg = _norm(sd, "policy_head.model.3", lg)
    logp = torch.log_softmax(lg.flatten(1), dim=1)
    w1 = sd["value_head.ffn.0.weight"].double()
    w1 = torch.cat((fmt.weight(w1[:, :64 * 256]), w1[:, 64 * 256:]), dim=1)
    hid = (torch.cat((y.flatten(1), meta), dim=1) @ w1.T + sd["value_head.ffn.0.bias"].double()).clamp_min(0)
    v = torch.tanh(hid @ sd["value_head.ffn.2.weight"].double().T + sd["value_head.ffn.2.bias"].double())
    return logp.numpy(), (v[:, 0] * (meta[:, 0] * 2 - 1)).numpy()


def run_heads(fmt, nets, games, monkeypatch, tag):
    """After the whole tower, t and y are the head GEMMs' inputs: forward_only's log-probs and values must match a
    float64 head on them at the fp32 tolerances.  n <= 128 finishes the value head inside the value-FC GEMM, larger
    batches in a separate kernel."""
    import net

    sd, blob, _ = nets[tag]
    e = _engine(blob, monkeypatch, mode=fmt.mode)
    try:
        for n in (37, 333):
            pos, _, _ = _batch(games, n)
            planes, meta = e.encode_only(pos)
            _, t, y = e.debug_tower(pos, len(_layers(sd)), 0)
            lp, v = e.forward_only(net.planes_i8_hwc_to_nchw(planes).numpy(), meta.astype(np.float32))
            lp_ref, v_ref = _heads_reference(fmt, sd, _nhwc_to_nchw(fmt.decode(t)), _nhwc_to_nchw(fmt.decode(y)),
                                             torch.from_numpy(meta).double())
            dl, dv = float(np.abs(lp - lp_ref).max()), float(np.abs(v - v_ref).max())
            print(f"{fmt.name} {tag} heads n={n}: max |d logp| {dl:.2e}  max |d value| {dv:.2e}")
            assert dl <= 1e-4 and dv <= 1e-5, (tag, n, dl, dv)
    finally:
        e.close()


@pytest.mark.parametrize("tag", ["n2", "n19", "bn_se", "stress"])
def test_heads_from_tower_buffers(nets, games, monkeypatch, tag):
    run_heads(BF16, nets, games, monkeypatch, tag)


# ---- the stress net end to end ----------------------------------------------------------------------------------
def test_stress_net_end_to_end(co, nets, games, monkeypatch):
    """Shifted conv biases, negative gammas, large betas and saturated SE gates: every mode against the oracle."""
    import net

    sd, blob, _ = nets["stress"]
    gs, depths = games[0][:161], games[1][:161]
    pos, moves, off, mv_all = games_to_batch(gs, depths)
    planes = np.stack([g.encode(dp)[0] for g, dp in zip(gs, depths)])
    meta = np.stack([g.encode(dp)[1] for g, dp in zip(gs, depths)])
    lp, v = net.forward(sd, net.planes_i8_hwc_to_nchw(planes), torch.from_numpy(meta).float())
    ref = np.concatenate([co.post_process(lp[i].numpy(), g.move_indices(mv)) for i, (g, mv) in enumerate(zip(gs, mv_all))])
    vref = v.numpy().reshape(-1)
    bad = []
    for mode, tol in ((scb200.SC_MODE_BF16, 2e-2), (scb200.SC_MODE_FP32, 1e-4), (scb200.SC_MODE_FP32_FFMA, 1e-4)):
        e = _engine(blob, monkeypatch, max_batch=256, mode=mode)
        try:
            pri, val = e.eval(pos, moves, off)
            p1, v1 = e.eval(pos[:1], moves[: off[1]], off[:2])
        finally:
            e.close()
        dp, dv = float(np.abs(pri - ref).max()), float(np.abs(val - vref).max())
        d1 = max(float(np.abs(p1 - ref[: off[1]]).max()), abs(float(v1[0]) - float(vref[0])))
        print(f"stress mode={mode}: max |d prior| {dp:.2e}  max |d value| {dv:.2e}  one leaf {d1:.2e}")
        if not (dp < tol and dv < tol and d1 < tol):
            bad.append((mode, dp, dv, d1))
    assert not bad, bad


# ---- launch variants and drivers of the fp16 and fp8 modes (test_gpu_fp16, test_gpu_fp8) ------------------------
LAUNCH_VARIANTS = [{"SCB200_TOWER": "0"}, {"SCB200_TOWER_GROUP": "0"}, {"SCB200_FUSE_GATHER": "0"},
                   {"SCB200_FUSE_VALUE": "0"}]


def check_launch_variant(mode, net19, batch2048, monkeypatch, env):
    """Per-layer launches, other tile groupings and the stand-alone value tail give the same bits as the defaults, on
    the throughput kernels.  The stand-alone legal-move gather (policy.cu) is the fused epilogue's arithmetic in another
    kernel, not the same instruction sequence: as in bf16 mode (test_fused_policy_gather_matches_standalone_kernel) the
    values are bit-equal and the priors agree to 2e-6."""
    games, pos, moves, off, mv_all, lp, v, pri_ref = batch2048
    for n in (2048, 100):
        a = _eval(net19[1], monkeypatch, pos[:n], moves[: off[n]], off[: n + 1], env={"SCB200_LATENCY": "0"}, mode=mode)
        b = _eval(net19[1], monkeypatch, pos[:n], moves[: off[n]], off[: n + 1], env=dict(env, SCB200_LATENCY="0"),
                  mode=mode)
        assert np.array_equal(a[1], b[1]), (env, n)
        if "SCB200_FUSE_GATHER" in env:
            assert np.abs(a[0] - b[0]).max() < 2e-6, (env, n)
        else:
            assert np.array_equal(a[0], b[0]), (env, n)


def check_selfplay_arena_and_game(mode, co, nets, monkeypatch):
    """Self-play twice with the same seed gives the same traces of legal moves, game_selfplay mirrors its first game,
    and an arena against a bf16 engine completes."""
    blob = nets["n2"][1]
    eng = _engine(blob, monkeypatch, max_batch=64, mode=mode)
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
