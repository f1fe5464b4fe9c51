"""Every layer of the two fp32 modes against a float64 reference of the same layer (sc_debug_tower_f32): the bf16x3
split mode SC_MODE_FP32 (tc_gemm_kernel EPI_F32, split3_store, ln_f32_kernel, se_res_f32_kernel) and its FFMA referee
SC_MODE_FP32_FFMA (gemm_f32_kernel).

Every fp32 gate of the suite runs on SC_MODE_FP32, and the end-to-end bars (1e-4 against the oracle, 5e-5 against the
referee) cannot see a split GEMM that lost one or two of its six plane products: a float64 emulation of the 19-block
net with a2*b0 or a0*b2 dropped moves the log-probs by about 2e-5.  Here each layer starts from the kernel's own fp32
inputs (the buffers of the previous n_layers call) and is compared with float64 arithmetic of that one layer on the
unrounded fp32 weights.  Notation: u = 2^-24 (fp32's unit roundoff); per output element
S = conv(|x|, |w|) + |b| in float64; per square sigma = sqrt(var + eps), z^ = (a - mean) / sigma, M = max |a|.

(a) The dense bound.
  * Convolution + bias: |da| <= c u S with c = C_CONV = 16.  This is not a worst case (one ulp per addition of 2304 x 6
    products would be thousands of u S) but a measured scale: torch's fp32 CPU convolution of three 19-block layers is
    at most 5.25 u S from float64; the tensor-core and the FFMA accumulation orders differ from it.  (First B200 run,
    1000 W power limit: every layer of both modes at 0.05 .. 0.51 of the whole bound below.)
  * LayerNorm: da moves z by |gamma| da / sigma.  ln_f32_kernel's two-pass mean sums each lane's 8 channels in order
    (partial sums up to 2M .. 8M: 35 M per lane, 1120 M for 32 lanes) and then the lanes in a 31-addition butterfly
    (16 x 16M + 8 x 32M + 4 x 64M + 2 x 128M + 256M = 1280 M), so the sum is off by at most 2400 u M, the mean by
    2400 / C u M plus its own rounding (u M when C is not a power of two; kept for all C): LN_MEAN = 2400 / 256 + 1.
    A shifted mean shifts every a - mean alike: |gamma| LN_MEAN u M / sigma.  This term is what carries the stress net's
    conv biases shifted by 300x / 5000x the square's spread (the bf16 test derives its own for the bf16 kernels); on
    ordinary layers M / sigma is a few and the term is small.  rstd: the sum of squares (13 additions of positive terms:
    13 u relative), eps and rsqrtf (2 ulp) give 11 u relative; d * rstd * gamma + beta adds two roundings relative to
    gamma z^ and one relative to z.  In all
        tol_z = |gamma| u (c S + LN_MEAN M) / sigma + 16 u |gamma z^| + 2 u |z|,
    and tol_z = c u S for folded-BatchNorm layers (no normalisation).  ReLU does not increase an error.
  * SE + residual (se_res_f32_kernel, out = relu(fmaf(g, z, x))): the pool sums 64 squares in order (63 u sum |z|, then
    * 1/64 exact), fc1 and fc2 are fma chains of 256 and 128 terms on their bias (n u sum |terms| each), g =
    1 / (1 + expf(-p)) adds 8 u g.  Propagated: dm = mean(tol_z) + 64 u mean |z|; dh = |W1| dm + 257 u (|b1| + |W1||m|);
    dp = |W2| dh + 129 u (|b2| + |W2||h|); dg = g (1 - g) dp + 8 u g; and
        tol_x = g tol_z + dg |z| + u |out|
    (g = 1, dg = 0 for residual-only blocks).  conv2 writes z to y and out to x; both are checked.
  Every element of every written buffer must be within its bound, and every buffer a layer does not write must be
  unchanged.  max err / bound is printed per layer.

(b) Sparse exact nets.  The dense bound separates a dropped product from accumulation noise by only about 2x, so
2-block BatchNorm nets without SE hold the split to ulps: each output channel of every convolution has k in {1, 2}
non-zero folded weights of magnitude 0.25 .. 1 whose mid and lo bf16 planes are at least 2^-10 and 2^-18 of the weight
(so each of the six products is far above the bound below), folded biases below 0.1, on distinct taps, spread over
all 9 taps (every padding edge), every 64-channel K chunk and both 64-plane chunks of the stem (its pawn planes, the
densest ones).  With the BatchNorm folded there is no normalisation: a layer is relu(sum x w + b), which float64
gives exactly from the few products.  Bound (12 k + 2) u (sum |x w| + |b|): the kernel makes 6 k accumulator additions
of non-zero products, each off by at most one ulp (2 u) of a partial sum <= sum |x w|, rounding or truncating, and one
more at the bias; the three products the split drops (i + j > 2) are <= 2 u |x w| per weight together, less than the
count over-charges (five of each weight's six products are <= 2^-7 |x w| and the first weight's additions happen on an
accumulator that holds only them).  conv2's relu(y + x) adds u |out|.

(c) Planes, bit for bit: every layer that emits operand planes (stem and conv2: x's, conv1: t's) must emit
hi = RN_bf16(x), mid = RN_bf16(x - hi), lo = RN_bf16(x - hi - mid), and hi + mid + lo == x exactly, for every element
of rows 0 .. n - 1 of the returned fp32 buffer.

(d) Heads.  After the whole tower t and y are the inputs of the policy GEMM (gemm_f32 256 -> 73, ln_f32 with C = 73,
ld = 80, log-softmax) and the value FC (gemm_f32 split-K 16, value_finish_kernel<false>); forward_only must match
float64 heads computed on them within |d log-prob| <= 1e-5 and |d value| <= 2e-6.  Size of the errors: a logit is a
256-term fma chain whose rounding errors are independent, about sqrt(256) u x the partial sums' size (~0.5), 5e-7;
through LN(73) (1 / sigma ~ 2, |gamma| <= 1.5) and log-softmax (the max-subtracted sum of 4672 exps: ~12 u relative,
times 2 for the shift of every entry) that is ~2e-6.  The value is tanh of 128 hidden units of 16384-term sums taken
as 16 ordered chains of 1024: ~sqrt(16384) u |partials| ~ 1e-6 relative per unit, ~1e-7 .. 5e-7 on the value.  The
bars leave 5x over those estimates and are 10x / 5x below the end-to-end gates, where a head that reads a rounded
buffer or a wrong LayerNorm width fails by orders of magnitude.  (First B200 run, 1000 W power limit, both modes:
2.8e-6 .. 3.8e-6 on the log-probs, 1.5e-7 .. 3.6e-7 on the values.)

(e) CPU checks that the bounds catch real bugs (no GPU): on the sparse nets' first three layers a float64 emulation of
the documented arithmetic (the six products smallest first, fp32 round-to-nearest after each addition, then + bias)
passes (b)'s bound, and dropping any one product, a two-plane split or planes rounded from the wrong residual exceeds
it on >= 10 % of the live elements (those some non-zero product reaches and that are not zero on both sides after
the ReLU).  The stem has one A plane (its 0/1 inputs are exact in bf16) and three products:
dropping a product with a1 or a2 is no change there, so only the three it has are dropped.  On n2 and stress the dense
bound rejects LayerNorm eps = 1e-5 instead of 1e-6, the SE pool divided by 63 and the gate applied after the residual,
and admits a plain fp32 evaluation of each layer on the CPU.
"""
import types

import numpy as np
import pytest
import scb200
import torch
import torch.nn.functional as F
from scb200.export import BN_EPS

import test_gpu_layer_reference as tlr
from test_gpu_layer_reference import (PLANES, X, T, Y, _batch, _engine, _engine_tensors, _heads_reference, _layers,
                                      _nhwc_to_nchw, _norm, games, nets)  # noqa: F401  (fixtures)

U = 2.0 ** -24
C_CONV = 16
LN_MEAN = 2400 / 256 + 1
PX, PT = 3, 4                      # sc_debug_tower_f32's operand-plane buffers
BUF_NAMES = ("x", "t", "y", "px", "pt")
BOARDS_333 = [0, 1, 2, 3, 4, 5, 127, 128, 200, 329, 330, 331, 332]
EXACT = types.SimpleNamespace(weight=lambda w: w.double())   # _heads_reference's weights: fp32, unrounded
MODES = {"split": scb200.SC_MODE_FP32, "ffma": scb200.SC_MODE_FP32_FFMA}


# ---- float64 layer and its dense bound --------------------------------------------------------------------------
def _layer64(sd, layer, inp, resid, pool=64.0, gate_after_residual=False):
    """One fp32-mode layer in float64 on NCHW inputs with the unrounded fp32 weights: a dict with a = conv + bias,
    S = conv(|x|, |w|) + |b|, z = norm(a), out = what the layer writes last (x for conv2), and the SE pieces.  `pool` and
    `gate_after_residual` are mutants for (e)."""
    conv, norm, _, _, relu, se = layer
    w, b = sd[conv + ".weight"].double(), sd[conv + ".bias"].double()
    pad = w.shape[-1] // 2
    r = {"a": F.conv2d(inp, w, b, padding=pad), "S": F.conv2d(inp.abs(), w.abs(), b.abs(), padding=pad)}
    r["z"] = z = _norm(sd, norm, r["a"])
    if se is None:
        r["out"] = z.clamp_min(0) if relu else z
        return r
    if se == "residual":
        g = torch.ones(z.shape[0], z.shape[1], 1, 1, dtype=torch.float64)
    else:
        r["m"] = m = z.sum(dim=(2, 3)) / pool
        r["w1"], r["b1"] = sd[se + "fc1.weight"].double().reshape(128, 256), sd[se + "fc1.bias"].double()
        r["w2"], r["b2"] = sd[se + "fc2.weight"].double().reshape(256, 128), sd[se + "fc2.bias"].double()
        r["h"] = h = (m @ r["w1"].T + r["b1"]).clamp_min(0)
        g = torch.sigmoid(h @ r["w2"].T + r["b2"])[:, :, None, None]
    r["g"] = g
    r["out"] = (g * (z + resid) if gate_after_residual else g * z + resid).clamp_min(0)
    return r


def _dense_bound(sd, layer, r):
    """(tol of the first buffer written: z / relu(z), tol of conv2's x or None), the module docstring's (a)"""
    _, norm, _, _, _, se = layer
    if norm + ".weight" in sd:
        a = r["a"]
        gam = sd[norm + ".weight"].double().abs().view(1, -1, 1, 1)
        sigma = torch.sqrt(a.var(dim=1, unbiased=False, keepdim=True) + tlr.LN_EPS)
        zhat = (a - a.mean(dim=1, keepdim=True)) / sigma
        big_m = a.abs().amax(dim=1, keepdim=True)
        tol_z = gam * U * (C_CONV * r["S"] + LN_MEAN * big_m) / sigma + 16 * U * (gam * zhat).abs() + 2 * U * r["z"].abs()
    else:
        tol_z = C_CONV * U * r["S"]
    if se is None:
        return tol_z, None
    z, g = r["z"], r["g"]
    if se == "residual":
        dg = torch.zeros_like(g)
    else:
        dm = tol_z.mean(dim=(2, 3)) + 64 * U * z.abs().mean(dim=(2, 3))
        aw1, aw2 = r["w1"].abs(), r["w2"].abs()
        dh = dm @ aw1.T + 257 * U * (r["b1"].abs() + r["m"].abs() @ aw1.T)
        dp = dh @ aw2.T + 129 * U * (r["b2"].abs() + r["h"].abs() @ aw2.T)
        gg = g[:, :, 0, 0]
        dg = (gg * (1 - gg) * dp + 8 * U * gg)[:, :, None, None]
    return tol_z, g * tol_z + dg * z.abs() + U * r["out"].abs()


def _written(layer, split):
    """buffers a layer writes, in sc_debug_tower_f32's numbering (PX / PT: the operand planes of x / t)"""
    conv, _, reads, writes, _, se = layer
    out = {writes} if se is None else {X, Y}
    if split and (reads == PLANES or se is not None):
        out.add(PX)
    if split and conv.endswith(".conv1"):
        out.add(PT)
    return out


def _split3_bits(x):
    """fp32 [..., 256] -> the three bf16 planes [..., 768] split3_store writes (hi, mid, lo from successive exact
    residuals, round to nearest even), as uint16"""
    t = torch.from_numpy(np.ascontiguousarray(x))
    hi = t.to(torch.bfloat16)
    r = t - hi.float()                   # exact: x and hi agree in their leading bits
    mid = r.to(torch.bfloat16)
    lo = (r - mid.float()).to(torch.bfloat16)
    return torch.cat((hi, mid, lo), dim=-1).view(torch.int16).numpy().view(np.uint16)


def _check_planes(x, planes, what):
    """(c): the returned planes are split3 of the returned fp32 buffer bit for bit, and add up to it exactly"""
    want = _split3_bits(x)
    bad = np.argwhere(planes != want)
    assert bad.size == 0, f"{what}: {len(bad)} plane elements differ, first at {tuple(bad[0])}: " \
                          f"got {planes[tuple(bad[0])]:#06x} want {want[tuple(bad[0])]:#06x}"
    v = tlr._bf16_bits_to_f64(planes.reshape(-1, 3, 256).transpose(1, 0, 2).copy()).sum(dim=0)
    assert torch.equal(v, torch.from_numpy(x.reshape(-1, 256)).double()), f"{what}: hi + mid + lo != x"


# ---- the per-layer walk ------------------------------------------------------------------------------------------
def _walk_layers(tag, sd, e, pos, reference, boards=None):
    """Runs k = 1 .. L layers and checks layer k from the k - 1 call's buffers: untouched buffers unchanged, the
    written ones against `reference(layer, inp, resid)` -> [(buffer, float64 value, bound)], emitted planes bit-exact."""
    import net

    split = e.mode == scb200.SC_MODE_FP32
    n = len(pos)
    boards = np.arange(n) if boards is None else np.asarray(boards)
    planes, _ = e.encode_only(pos)
    prev = [np.zeros((n, 64, 256), np.float32) for _ in range(3)] + \
           [np.zeros((n, 64, 768), np.uint16) if split else None for _ in range(2)]
    prev_planes = net.planes_i8_hwc_to_nchw(planes[boards]).double()
    name = f"{'split' if split else 'ffma'} {tag} n={n}"
    failures, ratios = [], []
    for k, layer in enumerate(_layers(sd), start=1):
        cur = e.debug_tower_f32(pos, k, planes=split)
        conv, _, reads, _, _, se = layer
        written = _written(layer, split)
        for b in range(5):
            if b not in written and cur[b] is not None:
                assert np.array_equal(cur[b], prev[b]), f"{name} layer {k} ({conv}) changed buffer {BUF_NAMES[b]}"
        inp = prev_planes if reads == PLANES else _nhwc_to_nchw(torch.from_numpy(prev[reads][boards]).double())
        resid = _nhwc_to_nchw(torch.from_numpy(prev[X][boards]).double()) if se is not None else None
        worst = 0.0
        for b, ref, tol in reference(layer, inp, resid):
            got = _nhwc_to_nchw(torch.from_numpy(cur[b][boards]).double()).numpy()
            ref, tol = ref.numpy(), tol.numpy()
            assert np.isfinite(got).all(), f"{name} layer {k} ({conv}): non-finite output"
            err = np.abs(got - ref)
            worst = max(worst, float(np.max(err / np.maximum(tol, 1e-300))))
            if not (err <= tol).all():
                i = np.unravel_index(np.argmax(err / np.maximum(tol, 1e-300)), err.shape)
                failures.append(f"layer {k} ({conv}) buffer {BUF_NAMES[b]}: {int((err > tol).sum())} elements out of "
                                f"bound, worst at (board {boards[i[0]]}, c {i[1]}, sq {i[2] * 8 + i[3]}): got {got[i]:.9g} "
                                f"ref {ref[i]:.9g} err {err[i]:.3g} bound {tol[i]:.3g}")
        print(f"{name} layer {k:2d} {conv:22s} max err / bound {worst:7.4f}")
        ratios.append(worst)
        for b, src in ((PX, X), (PT, T)):
            if b in written:
                _check_planes(cur[src], cur[b], f"{name} layer {k} ({conv}) planes {BUF_NAMES[b]}")
        prev = cur
    print(f"{name}: max err / bound over the layers {min(ratios):.4f} .. {max(ratios):.4f}")
    assert not failures, f"{name}:\n" + "\n".join(failures)


def _dense_reference(sd):
    def ref(layer, inp, resid):
        r = _layer64(sd, layer, inp, resid)
        tol_z, tol_x = _dense_bound(sd, layer, r)
        if tol_x is None:
            return [(layer[3], r["out"], tol_z)]
        return [(Y, r["z"], tol_z), (X, r["out"], tol_x)]
    return ref


def _run_dense(tag, nets, games, monkeypatch, mode, sizes, boards=BOARDS_333, max_batch=512):
    sd, blob, _ = nets[tag]
    e = _engine(blob, monkeypatch, max_batch=max_batch, mode=mode)
    try:
        for n in sizes:
            pos, _, _ = _batch(games, n)
            _walk_layers(tag, sd, e, pos, _dense_reference(sd))
        if boards is not None:
            pos, _, _ = _batch(games, 333)
            _walk_layers(tag, sd, e, pos, _dense_reference(sd), boards=boards)
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["n2", "stress"])
def test_split_layers(nets, games, monkeypatch, tag):
    """Partial CTA-pair tiles (a pair is 4 boards), several tile groups ending in a partial tile, and an engine with
    max_batch = 5 at n = 5, whose last 4-board tile runs past the 6 allocated boards."""
    _run_dense(tag, nets, games, monkeypatch, scb200.SC_MODE_FP32, (1, 2, 3, 5, 6))
    _run_dense(tag, nets, games, monkeypatch, scb200.SC_MODE_FP32, (5,), boards=None, max_batch=5)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["n19", "bn_se", "ln_nose", "bn_nose"])
def test_split_layers_other_nets(nets, games, monkeypatch, tag):
    """All 41 layers of the 19-block seed-0 net, and the folded-BatchNorm / residual-only variants."""
    _run_dense(tag, nets, games, monkeypatch, scb200.SC_MODE_FP32, (3,), boards=None, max_batch=16)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["n2", "stress", "n19"])
def test_ffma_referee_layers(nets, games, monkeypatch, tag):
    _run_dense(tag, nets, games, monkeypatch, scb200.SC_MODE_FP32_FFMA, (1, 3))


@pytest.mark.gpu
def test_debug_tower_f32_rejects_other_modes(nets, games, monkeypatch):
    pos, _, _ = _batch(games, 2)
    blob = nets["n2"][1]
    for mode in (scb200.SC_MODE_BF16, scb200.SC_MODE_FP16, scb200.SC_MODE_FP8):
        e = _engine(blob, monkeypatch, max_batch=16, mode=mode)
        try:
            with pytest.raises(scb200.SCError, match="sc_debug_tower_f32"):
                e.debug_tower_f32(pos, 1, planes=False)
        finally:
            e.close()
    e = _engine(blob, monkeypatch, max_batch=16, mode=scb200.SC_MODE_FP32_FFMA)
    try:
        with pytest.raises(scb200.SCError, match="operand planes"):
            e.debug_tower_f32(pos, 1, planes=True)
    finally:
        e.close()


# ---- sparse exact nets ------------------------------------------------------------------------------------------
PAWN_PLANES = [14 * h + s for h in range(8) for s in (0, 6)]   # the densest input planes, in both 64-plane chunks
SPARSE_SEEDS = {"sparse_a": 41, "sparse_b": 42}


def _planes_large(w32):
    """the mid and lo bf16 planes of w32 are at least 2^-10 / 2^-18 of it (all three non-zero, and a product dropped
    from the split moves the output by 32 .. 128 u |x w|: far outside (b)'s bound)"""
    _, mid, lo = tlr._bf16_bits_to_f64(_split3_bits(np.array([w32], np.float32))).abs().tolist()
    return mid >= 2.0 ** -10 * abs(float(w32)) and lo >= 2.0 ** -18 * abs(float(w32))


def _sparse_state_dict(seed):
    """2-block BatchNorm net without SE whose folded convolutions have k = 1 or 2 non-zero weights per output channel
    (module docstring, (b)); BatchNorm statistics near 1 so that the folded weights stay in 0.25 .. 1"""
    import net

    sd = net.init_variant_state_dict(2, seed, "BatchNorm", False)
    g = torch.Generator().manual_seed(seed)
    off = seed % 7
    for conv, norm, reads, _, _, _ in _layers(sd):
        cout, cin, kh, kw = sd[conv + ".weight"].shape
        taps = kh * kw
        gamma = 0.8 + 0.4 * torch.rand(cout, generator=g)
        var = 0.8 + 0.4 * torch.rand(cout, generator=g)
        sd[norm + ".weight"], sd[norm + ".running_var"] = gamma, var
        sd[norm + ".running_mean"] = 0.03 * (2 * torch.rand(cout, generator=g) - 1)   # folded bias: |b| < 0.1, so the
        sd[norm + ".bias"] = 0.05 * (2 * torch.rand(cout, generator=g) - 1)           # products dominate the bound
        scale = gamma.double() / torch.sqrt(var.double() + BN_EPS)
        w = torch.zeros(cout, cin, taps)
        for co in range(cout):
            for j in range(1 + (co + off) % 2):
                tap = (co + off + 4 * j) % taps          # two weights of a channel: distinct taps of a 3x3
                ci = PAWN_PLANES[(co * 5 + j * 3 + off) % 16] if reads == PLANES else (co * 67 + j * 101 + off) % cin
                while True:                              # the folded weight's mid and lo planes not small
                    t = float(torch.rand(1, generator=g)) * 0.65 + 0.3
                    t = -t if torch.rand(1, generator=g) < 0.5 else t
                    raw = np.float32(t / float(scale[co]))
                    if _planes_large(np.float32(float(raw) * float(scale[co]))):
                        break
                w[co, ci, tap] = float(raw)
        sd[conv + ".weight"] = w.reshape(cout, cin, kh, kw)
    return sd


@pytest.fixture(scope="module")
def sparse_nets(tmp_path_factory):
    """name -> (the folded tensors the engine loads, blob path)"""
    d = tmp_path_factory.mktemp("sparse")
    out = {}
    for name, seed in SPARSE_SEEDS.items():
        sd = _sparse_state_dict(seed)
        p = str(d / f"{name}.scw")
        scb200.write_blob(sd, p)
        out[name] = (_engine_tensors(sd), p)
    return out


def _sparse_terms(x, w):
    """x NCHW [n, cin, 8, 8], w [cout, cin, kh, kw] with few non-zeros -> (index of the output channel, tap, and the
    product x * w [nnz, n, 8, 8] of each non-zero weight), in float64"""
    kh = w.shape[-1]
    p = kh // 2
    xp = F.pad(x, (p, p, p, p))
    co, ci, ty, tx = w.nonzero(as_tuple=True)
    win = torch.stack([xp[:, c, a:a + 8, b:b + 8] for c, a, b in zip(ci.tolist(), ty.tolist(), tx.tolist())]) \
        if len(co) else torch.zeros(0, x.shape[0], 8, 8, dtype=torch.float64)
    return co, ty * kh + tx, win, w[co, ci, ty, tx].double()


def _sparse_layer(sd, layer, inp, resid):
    """float64 of a sparse layer and its (b) bound: [(buffer, value, bound)]"""
    conv, _, _, writes, relu, se = layer
    w, b = sd[conv + ".weight"], sd[conv + ".bias"].double()
    co, _, win, wv = _sparse_terms(inp, w)
    n, cout = inp.shape[0], w.shape[0]
    prod = win * wv.view(-1, 1, 1, 1)
    a = torch.zeros(cout, n, 8, 8, dtype=torch.float64).index_add_(0, co, prod).permute(1, 0, 2, 3)
    s = torch.zeros(cout, n, 8, 8, dtype=torch.float64).index_add_(0, co, prod.abs()).permute(1, 0, 2, 3)
    k = (w.reshape(cout, -1) != 0).sum(dim=1).double().view(1, -1, 1, 1)
    a = a + b.view(1, -1, 1, 1)
    tol = (12 * k + 2) * U * (s + b.abs().view(1, -1, 1, 1))
    if se is None:
        return [(writes, a.clamp_min(0) if relu else a, tol)]
    out = (a + resid).clamp_min(0)
    return [(Y, a, tol), (X, out, tol + U * out.abs())]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("tag", sorted(SPARSE_SEEDS))
def test_sparse_exact_layers(sparse_nets, games, monkeypatch, tag, mode):
    sd, blob = sparse_nets[tag]
    e = _engine(blob, monkeypatch, max_batch=512, mode=MODES[mode])
    try:
        for n in (1, 5, 333):
            pos, _, _ = _batch(games, n)
            _walk_layers(tag, sd, e, pos, lambda layer, inp, resid: _sparse_layer(sd, layer, inp, resid))
    finally:
        e.close()


# ---- heads ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", sorted(MODES))
@pytest.mark.parametrize("tag", ["n2", "n19", "stress"])
def test_heads_from_tower_buffers(nets, games, monkeypatch, tag, mode):
    """(d): forward_only's log-probs and values against float64 heads on the tower's own fp32 t and y."""
    import net

    sd, blob, _ = nets[tag]
    e = _engine(blob, monkeypatch, max_batch=512, mode=MODES[mode])
    try:
        for n in (37, 333):
            pos, _, _ = _batch(games, n)
            planes, meta = e.encode_only(pos)
            _, t, y, _, _ = e.debug_tower_f32(pos, 0, planes=False)
            lp, v = e.forward_only(net.planes_i8_hwc_to_nchw(planes).numpy(), meta.astype(np.float32))
            lp_ref, v_ref = _heads_reference(EXACT, sd, _nhwc_to_nchw(torch.from_numpy(t).double()),
                                             _nhwc_to_nchw(torch.from_numpy(y).double()), torch.from_numpy(meta).double())
            dl, dv = float(np.abs(lp - lp_ref).max()), float(np.abs(v - v_ref).max())
            print(f"{mode} {tag} heads n={n}: max |d logp| {dl:.2e}  max |d value| {dv:.2e}")
            assert dl <= 1e-5 and dv <= 2e-6, (mode, tag, n, dl, dv)
    finally:
        e.close()


# ---- (e) the bounds against known bugs, on the CPU -----------------------------------------------------------------
def _planes3(x, two_planes=False, wrong_residual=False):
    """hi, mid, lo of fp32 values (a float64 tensor holding fp32 numbers) as float64; mutants: lo = 0, or lo rounded
    from x - hi instead of x - hi - mid"""
    t = x.float()
    hi = t.to(torch.bfloat16).float()
    mid = (t - hi).to(torch.bfloat16).float()
    lo = ((t - hi) if wrong_residual else (t - hi - mid)).to(torch.bfloat16).float()
    if two_planes:
        lo = torch.zeros_like(lo)
    return [p.double() for p in (hi, mid, lo)]


SPLIT_PAIRS = [(0, 2), (1, 1), (2, 0), (0, 1), (1, 0), (0, 0)]   # tc_split_conv_create's order, smallest first


def _emulate_split(sd, layer, inp, resid, drop=None, **planes_kw):
    """The split GEMM's documented arithmetic on a sparse layer: per tap, the (A plane, B plane) products smallest
    first, each added to an fp32 accumulator with round-to-nearest (a channel's weights sit on distinct taps: one
    product per addition), then + bias in fp32; the layer's epilogue after it.  Input planes: one A plane (0/1)."""
    conv, _, reads, writes, relu, se = layer
    w, b = sd[conv + ".weight"], sd[conv + ".bias"].float()
    a_pl = [inp, torch.zeros_like(inp), torch.zeros_like(inp)] if reads == PLANES else _planes3(inp, **planes_kw)
    w_pl = _planes3(w.double(), **planes_kw)
    pairs = [(i, j) for i, j in SPLIT_PAIRS if (i, j) != drop]
    terms = {(i, j): _sparse_terms(a_pl[i], w_pl[j]) for i, j in pairs}
    n, cout = inp.shape[0], w.shape[0]
    acc = torch.zeros(n, cout, 8, 8, dtype=torch.float32)
    for t in range(w.shape[-1] * w.shape[-2]):
        for i, j in pairs:
            co, tap, win, wv = terms[(i, j)]
            keep = tap == t
            term = torch.zeros(cout, n, 8, 8, dtype=torch.float64).index_add_(
                0, co[keep], win[keep] * wv[keep].view(-1, 1, 1, 1)).permute(1, 0, 2, 3)
            acc = acc + term.float()                        # one product per channel and tap: term exact in fp32
    a = acc + b.view(1, -1, 1, 1)
    if se is None:
        return {writes: (a.clamp_min(0) if relu else a).double()}
    return {Y: a.double(), X: (a + resid.float()).clamp_min(0).double()}


def _sparse_chain(sd, planes_nchw, n_layers):
    """inputs of the first n_layers layers as the kernels see them: the float64 chain rounded to fp32 per layer"""
    bufs = {PLANES: planes_nchw}
    steps = []
    for layer in _layers(sd)[:n_layers]:
        resid = bufs.get(X) if layer[5] is not None else None
        steps.append((layer, bufs[layer[2]], resid))
        for b, v, _ in _sparse_layer(sd, layer, bufs[layer[2]], resid):
            bufs[b] = v.float().double()
    return steps


def _cpu_planes(games, n):
    import net

    gs, depths = games
    return net.planes_i8_hwc_to_nchw(np.stack([g.encode(dp)[0] for g, dp in zip(gs[:n], depths[:n])])).double()


def test_sparse_bound_admits_the_split_and_rejects_broken_splits(sparse_nets, games):
    """(e), sparse nets: the emulated split passes (b)'s bound; each mutant exceeds it on >= 10 % of the live elements
    of every one of the first three layers (stem, conv1, conv2 + residual)."""
    mutants = {f"drop a{i}*b{j}": {"drop": (i, j)} for i, j in SPLIT_PAIRS}
    mutants["two-plane split"] = {"two_planes": True}
    mutants["lo from x - hi"] = {"wrong_residual": True}
    bad = []
    for tag, (sd, _) in sparse_nets.items():
        for layer, inp, resid in _sparse_chain(sd, _cpu_planes(games, 48), 3):
            refs = _sparse_layer(sd, layer, inp, resid)
            emu = _emulate_split(sd, layer, inp, resid)
            # live: an element some non-zero product reaches, not zero on both sides after the ReLU
            w = sd[layer[0] + ".weight"].double()
            reached = F.conv2d(inp.abs(), w.abs(), padding=w.shape[-1] // 2) > 0
            worst = max(float((torch.abs(emu[b] - ref) / tol).max()) for b, ref, tol in refs)
            print(f"{tag} {layer[0]:22s} emulated split: max err / bound {worst:.3f}")
            if worst > 1:
                bad.append(f"{tag} {layer[0]}: the emulated split exceeds the bound ({worst:.3f})")
            for name, kw in mutants.items():
                if layer[2] == PLANES and "drop" in kw and kw["drop"][0] > 0:
                    continue                                 # the stem has one A plane: nothing to drop
                mut = _emulate_split(sd, layer, inp, resid, **kw)
                fracs = []
                for b, ref, tol in refs:
                    live = ((ref != 0) | (mut[b] != 0)) & reached
                    fracs.append(float(((torch.abs(mut[b] - ref) > tol) & live).sum() / live.sum()))
                print(f"{tag} {layer[0]:22s} {name:16s}: out of bound on {min(fracs):.3f} of the live elements")
                if min(fracs) < 0.10:
                    bad.append(f"{tag} {layer[0]}: mutant '{name}' out of bound on only {min(fracs):.3f}")
    assert not bad, "\n".join(bad)


def _fp32_layer(sd, layer, inp, resid):
    """the layer in plain fp32 on the CPU (torch's convolution, a textbook LayerNorm and SE)"""
    conv, norm, _, _, relu, se = layer
    w, b = sd[conv + ".weight"].float(), sd[conv + ".bias"].float()
    a = F.conv2d(inp.float(), w, b, padding=w.shape[-1] // 2)
    if norm + ".weight" in sd:
        mean = a.mean(dim=1, keepdim=True)
        d = a - mean
        rstd = torch.rsqrt((d * d).mean(dim=1, keepdim=True) + tlr.LN_EPS)
        z = d * rstd * sd[norm + ".weight"].float().view(1, -1, 1, 1) + sd[norm + ".bias"].float().view(1, -1, 1, 1)
    else:
        z = a
    if se is None:
        return [(z.clamp_min(0) if relu else z).double()]
    g = torch.ones(1)
    if se != "residual":
        m = z.mean(dim=(2, 3))
        h = (m @ sd[se + "fc1.weight"].float().reshape(128, 256).T + sd[se + "fc1.bias"].float()).clamp_min(0)
        g = torch.sigmoid(h @ sd[se + "fc2.weight"].float().reshape(256, 128).T + sd[se + "fc2.bias"].float())
        g = g[:, :, None, None]
    return [z.double(), (g * z + resid.float()).clamp_min(0).double()]


def test_dense_bound_rejects_known_bugs(nets, games, monkeypatch):
    """(e), dense bound on n2 and stress: plain fp32 passes every layer; LayerNorm eps = 1e-5, the SE pool divided by
    63 and the gate applied after the residual each fail some layer by more than 2x the bound, so a kernel with the bug
    fails even where its own rounding error happens to pull toward the right value."""
    planes = _cpu_planes(games, 24)
    bad = []
    for tag in ("n2", "stress"):
        sd = nets[tag][0]
        bufs = {PLANES: planes}
        worst = {"fp32": 0.0, "eps 1e-5": 0.0, "pool / 63": 0.0, "gate after residual": 0.0}
        for layer in _layers(sd):
            inp, resid = bufs[layer[2]], (bufs[X] if layer[5] is not None else None)
            r = _layer64(sd, layer, inp, resid)
            tols = [t for t in _dense_bound(sd, layer, r) if t is not None]
            refs = [r["out"]] if layer[5] is None else [r["z"], r["out"]]

            def ratio(vals):
                return max(float((torch.abs(v - ref) / tol).max()) for v, ref, tol in zip(vals, refs, tols))

            worst["fp32"] = max(worst["fp32"], ratio(_fp32_layer(sd, layer, inp, resid)))
            with monkeypatch.context() as m:
                m.setattr(tlr, "LN_EPS", 1e-5)
                r_eps = _layer64(sd, layer, inp, resid)
            worst["eps 1e-5"] = max(worst["eps 1e-5"], ratio([r_eps["out"]] if layer[5] is None else
                                                              [r_eps["z"], r_eps["out"]]))
            if layer[5] is not None and layer[5] != "residual":
                r_pool = _layer64(sd, layer, inp, resid, pool=63.0)
                r_gate = _layer64(sd, layer, inp, resid, gate_after_residual=True)
                worst["pool / 63"] = max(worst["pool / 63"], ratio([r_pool["z"], r_pool["out"]]))
                worst["gate after residual"] = max(worst["gate after residual"], ratio([r_gate["z"], r_gate["out"]]))
            bufs[layer[3]] = r["out"].float().double()
        print(f"{tag}: max err / bound " + "  ".join(f"{k} {v:.3g}" for k, v in worst.items()))
        if worst.pop("fp32") > 1:
            bad.append(f"{tag}: plain fp32 exceeds the dense bound")
        bad += [f"{tag}: mutant '{k}' reaches only {v:.3g} x the bound" for k, v in worst.items() if v < 2]
    assert not bad, "\n".join(bad)
