"""sc_predict_stack: `Game::predict` for leaves given as move stacks, replayed and packed on the device.

The replay runs the host rules (csrc/host/chess_rules.hpp: Position::push, tkey, has_legal_ep, is_irreversible and the
shared repetition walk), so every packed leaf must equal the host's bit for bit: `scb200.rules_probe(history)`'s packed
leaf, with the slots from n_hist on zeroed and n_hist set (host::pack_position(g, n_hist)).  After the replay the call is
sc_predict, so moves, counts, priors and values must equal sc_predict's on the host-packed leaf with the host's
ep_square.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ("SC_MODE_FP32", "SC_MODE_BF16", "SC_MODE_FP32_FFMA", "SC_MODE_FP16")


def _sq(s):
    return (int(s[1]) - 1) * 8 + ord(s[0]) - ord("a")


def _uci(text):
    return [(_sq(u[:2]), _sq(u[2:4]), " pnbrqk".index(u[4]) if len(u) > 4 else 0) for u in text.split()]


# (moves, value of the last position in White's perspective)
FOOLS_MATE = (_uci("f2f3 e7e5 g2g4 d8h4"), -1.0)                                                # White is mated
SMOTHERED_MATE = (_uci("e2e4 e7e5 g1f3 b8c6 f1c4 c6d4 f3e5 d8g5 e5f7 g5g2 h1f1 g2e4 c4e2 d4f3"), -1.0)  # ... Nf3#
STALEMATE = (_uci("e2e3 a7a5 d1h5 a8a6 h5a5 h7h5 h2h4 a6h6 a5c7 f7f6 c7d7 e8f7 d7b7 d8d3 b7b8 d3h7 b8c8 f7g6 c8e6"), 0.0)

KNIGHTS = _uci("g1f3 g8f6 f3g1 f6g8")  # back to the start position every four plies


def _built_sequences():
    """Move lists whose repetition flags, castling rights and en-passant keys the packing depends on."""
    seqs = {
        "shuffle_5fold": KNIGHTS * 4 + _uci("g1f3"),
        "shuffle_pawn_break": KNIGHTS * 2 + _uci("e2e4") + _uci("g8f6 g1f3 f6g8 f3g1") * 3,
        "shuffle_capture_break": _uci("e2e4 d7d5") + _uci("g1f3 g8f6 f3g1 f6g8") * 2 + _uci("e4d5")
        + _uci("g8f6 g1f3 f6g8 f3g1") * 3,
        "shuffle_king_move": _uci("e2e4 e7e5") + KNIGHTS * 2 + _uci("e1e2 e8e7 e2e1 e7e8") * 3,
        "shuffle_rook_move": _uci("g1f3 g8f6 h1g1 h8g8 g1h1 g8h8") + _uci("b1c3 b8c6 c3b1 c6b8") * 3,
        # the bishop takes the rook on h8: Black loses its kingside right without moving the rook
        "rook_captured": _uci("b2b3 g7g5 c1b2 g8h6 b2h8") + _uci("b8c6 b1c3 c6b8 c3b1") * 3,
        # exd6 is legal: the key after d7d5 carries the en-passant square, the same board four plies on does not
        "ep_legal": _uci("e2e4 a7a6 e4e5 d7d5") + _uci("g1f3 g8f6 f3g1 f6g8") * 2,
        "ep_capture": _uci("e2e4 a7a6 e4e5 d7d5 e5d6"),
        # dxe3 is only pseudo-legal (the d4 pawn is pinned by Bb2 against Kf6): ep_square is e3, the key has none
        "ep_pinned": _uci("b2b3 d7d5 c1b2 d5d4 b1a3 f7f5 a3b1 e8f7 b1a3 f7f6 e2e4") + _uci("f6f7 a3b1 f7f6 b1a3") * 2,
        "fools_mate": FOOLS_MATE[0],
        "smothered_mate": SMOTHERED_MATE[0],
        "stalemate": STALEMATE[0],
    }
    # 300 reversible plies of rook moves after the opening pawn moves: the halfmove clock passes 150 (the 75-move rule)
    rooks = _uci("a2a4 a7a5 a1a3 a8a6")
    w, b = 0, 0
    for k in range(300):
        if k % 2 == 0:
            rooks.append((16 + w, 16 + (w + 1) % 8, 0))  # a3 .. h3 and round
            w = (w + 1) % 8
        else:
            rooks.append((40 + b, 40 + (b + 1) % 7, 0))  # a6 .. g6 and round
            b = (b + 1) % 7
    seqs["rook_shuffle_300"] = rooks
    return seqs


class StackLeaves:
    """Move stacks with the host's packed leaf (n_hist = min(8, plies + 1)), ep_square and legal moves."""

    def __init__(self):
        self.stacks, self.pos, self.ep, self.moves = [], [], [], []

    def add(self, hist):
        import scb200

        mv, pos, _ = scb200.rules_probe(hist)
        ep = -1
        if hist:
            f, t, _ = hist[-1]
            if (int(pos["slot"][0][0]) >> t) & 1 and abs(t - f) == 16:
                ep = (f + t) // 2
        self.stacks.append(list(hist))
        self.pos.append(pos)
        self.ep.append(ep)
        self.moves.append([tuple(int(x) for x in m) for m in mv])
        return mv

    def add_every_ply(self, hist):
        for k in range(len(hist) + 1):
            self.add(hist[:k])

    def positions(self, sl=slice(None)):
        import scb200

        return np.array(self.pos[sl], dtype=scb200.POSITION_DTYPE), np.array(self.ep[sl], dtype=np.int8)


def _expected(pos, n_hist):
    """host::pack_position(g, n_hist) from the packed leaf of the game-root history"""
    out = pos.copy()
    for i, h in enumerate(n_hist):
        out["slot"][i, h:] = 0
        out["n_hist"][i] = h
    return out


def _assert_packed_equal(got, exp, stacks):
    for i in range(len(got)):
        if got[i].tobytes() != exp[i].tobytes():
            raise AssertionError(f"leaf {i} ({len(stacks[i])} plies) packs differently: got {got[i]} expected {exp[i]}")


@pytest.fixture(scope="module")
def blob(tmp_path_factory):
    import net
    import scb200

    p = str(tmp_path_factory.mktemp("predict_stack") / "w.scw")
    scb200.write_blob(net.perturb_norm_params(net.init_state_dict(2, 7), 1234), p)
    return p


@pytest.fixture(scope="module")
def engine(blob):
    import scb200

    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 2048)
    yield e
    e.close()


@pytest.fixture(scope="module")
def random_leaves():
    """20 000 positions of seeded uniform random play, games of up to 300 plies (terminal positions included)."""
    lv = StackLeaves()
    rng = np.random.RandomState(17)
    while len(lv.pos) < 20000:
        hist = []
        for _ in range(301):
            mv = lv.add(hist)
            if len(mv) == 0 or len(lv.pos) >= 20000 or len(hist) == 300:
                break
            hist.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
    return lv


@pytest.fixture(scope="module")
def built_leaves():
    lv = StackLeaves()
    for seq in _built_sequences().values():
        lv.add_every_ply(seq)
    return lv


def _check_packing(engine, lv, n_hist=None):
    n_all = len(lv.pos)
    for b in range(0, n_all, engine.max_batch):
        sl = slice(b, min(n_all, b + engine.max_batch))
        stacks = lv.stacks[sl]
        nh = None if n_hist is None else n_hist[sl]
        moves, cnt, _, _, pos = engine.predict_stack(stacks, n_hist=nh, positions=True)
        host, _ = lv.positions(sl)
        exp = _expected(host, nh if nh is not None else [min(8, len(s) + 1) for s in stacks])
        _assert_packed_equal(pos, exp, stacks)
        for i, m in enumerate(lv.moves[sl]):
            assert cnt[i] == len(m) and [tuple(int(x) for x in (r["from"], r["to"], r["promo"])) for r in moves[i, : cnt[i]]] == m
    return n_all


def test_packing_matches_host_on_sample_games(engine, sample_games):
    lv = StackLeaves()
    for game in sample_games["games"]:
        lv.add_every_ply(_uci(game["uci"]))
    assert _check_packing(engine, lv) > 3500


def test_packing_matches_host_on_random_play(engine, random_leaves):
    lv = random_leaves
    assert max(len(s) for s in lv.stacks) == 300 and sum(e >= 0 for e in lv.ep) > 200
    assert sum(int(p["slot"][0][7]) & 1 for p in lv.pos) > 0  # repetitions occur
    assert _check_packing(engine, lv) == 20000


def test_packing_matches_host_for_every_n_hist(engine, random_leaves, built_leaves):
    lv = StackLeaves()
    for src in (random_leaves, built_leaves):
        for i in range(0, len(src.pos), max(1, len(src.pos) // 600)):
            lv.stacks.append(src.stacks[i])
            lv.pos.append(src.pos[i])
            lv.ep.append(src.ep[i])
            lv.moves.append(src.moves[i])
    rng = np.random.RandomState(5)
    for h in range(1, 9):
        nh = np.array([min(h, len(s) + 1) for s in lv.stacks], dtype=np.int8)
        _check_packing(engine, lv, nh)
    nh = np.array([rng.randint(1, min(8, len(s) + 1) + 1) for s in lv.stacks], dtype=np.int8)
    _check_packing(engine, lv, nh)


def test_packing_matches_host_on_built_sequences(engine, built_leaves):
    lv = built_leaves
    reps = [int(p["slot"][0][7]) for p in lv.pos]
    assert 3 in reps and 1 in reps  # three- and two-fold repetitions
    assert max(int(p["meta"][6]) for p in lv.pos) > 150  # past the 75-move clock
    seqs = _built_sequences()
    pinned = len(seqs["ep_pinned"]) - 8  # the position after e2e4: python-chess ep_square e3
    i = lv.stacks.index(seqs["ep_pinned"][:pinned])
    assert lv.ep[i] == 20
    _check_packing(engine, lv)
    # the same leaves one per call: the pinned staging buffer with the replay reading its own copy
    for k in range(0, len(lv.pos), 97):
        _, _, _, _, pos = engine.predict_stack([lv.stacks[k]], positions=True)
        exp = _expected(lv.positions(slice(k, k + 1))[0], [min(8, len(lv.stacks[k]) + 1)])
        _assert_packed_equal(pos, exp, lv.stacks[k : k + 1])


@pytest.mark.parametrize("mode", MODES)
def test_outputs_equal_sc_predict(blob, random_leaves, mode):
    """n = 1 / 37 (pinned staging; bf16/fp16: latency kernel), 129 (device buffers) and 2048 (throughput kernel)."""
    import scb200

    e = scb200.Engine(blob, 0, getattr(scb200, mode), 2048)
    lv = random_leaves
    flat_all = None
    for n in (1, 37, 129, 2048):
        for start in (0, 7000):
            sl = slice(start, start + n)
            pos, ep = lv.positions(sl)
            a = e.predict(pos, ep)
            if n == 129:  # the (flat array, offsets) form
                stacks = lv.stacks[sl]
                off = np.zeros(n + 1, dtype=np.int32)
                off[1:] = np.cumsum([len(s) for s in stacks])
                flat_all = np.zeros(int(off[-1]), dtype=scb200.MOVE_DTYPE)
                for s, o in zip(stacks, off[:-1]):
                    for k, m in enumerate(s):
                        flat_all[o + k] = (m[0], m[1], m[2], 0)
                b = e.predict_stack((flat_all, off))
            else:
                b = e.predict_stack(lv.stacks[sl])
            cnt = a[1]
            assert np.array_equal(cnt, b[1]), (mode, n)
            for i in range(n):
                c = int(cnt[i])
                assert np.array_equal(a[0][i, :c].view(np.uint32), b[0][i, :c].view(np.uint32)), (mode, n, i)
                assert np.array_equal(a[2][i, :c].view(np.uint32), b[2][i, :c].view(np.uint32)), (mode, n, i)
            assert np.array_equal(a[3].view(np.uint32), b[3].view(np.uint32)), (mode, n)
    assert flat_all is not None
    # terminal leaves reached by a move list get predict's terminal value, alone and in a batch
    terminal = (FOOLS_MATE, SMOTHERED_MATE, STALEMATE)
    stacks = [s for s, _ in terminal] + [[]]
    _, cnt, _, val = e.predict_stack(stacks)
    assert cnt.tolist() == [0, 0, 0, 20] and val[:3].tolist() == [v for _, v in terminal]
    for s, v in terminal:
        _, c1, _, v1 = e.predict_stack([s])
        assert c1[0] == 0 and v1[0] == v
    e.close()


def _raw_predict_stack(engine, flat, off, n_hist=None, guard_rows=1):
    """sc_predict_stack through ctypes with guard rows past the n output rows, to see every byte the call writes."""
    import scb200

    n = len(off) - 1
    rows = n + guard_rows
    pos = np.full(rows, 0x5A, dtype=np.uint8).repeat(scb200.POSITION_DTYPE.itemsize).view(scb200.POSITION_DTYPE).copy()
    moves = np.full((rows, scb200.SC_MAX_MOVES), 0xAB, dtype=np.uint32)
    cnt = np.full(rows, -7, dtype=np.int32)
    priors = np.full((rows, scb200.SC_MAX_MOVES), 7.0, dtype=np.float32)
    vals = np.full(rows, 7.0, dtype=np.float32)
    flat = np.ascontiguousarray(flat, dtype=scb200.MOVE_DTYPE)
    off = np.ascontiguousarray(off, dtype=np.int32)
    nh = None if n_hist is None else np.ascontiguousarray(n_hist, dtype=np.int8)
    rc = scb200.load_library().sc_predict_stack(
        engine.handle, n, flat.ctypes.data if len(flat) else None, off.ctypes.data, None if nh is None else nh.ctypes.data,
        pos.ctypes.data, moves.ctypes.data, cnt.ctypes.data, priors.ctypes.data, vals.ctypes.data, None)
    assert (pos[n:].view(np.uint8) == 0x5A).all()
    assert (moves[n:] == 0xAB).all() and (cnt[n:] == -7).all() and (priors[n:] == 7.0).all() and (vals[n:] == 7.0).all()
    return rc, pos[:n], moves[:n].view(scb200.MOVE_DTYPE), cnt[:n], vals[:n]


def _flat(stacks):
    import scb200

    off = np.zeros(len(stacks) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(s) for s in stacks])
    flat = np.zeros(int(off[-1]), dtype=scb200.MOVE_DTYPE)
    for s, o in zip(stacks, off[:-1]):
        for k, m in enumerate(s):
            flat[o + k] = (m[0], m[1], m[2], 0)
    return flat, off


def test_bad_arguments(blob, random_leaves):
    import scb200

    L = scb200.load_library()
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 8)
    stacks = random_leaves.stacks[100:108]
    flat, off = _flat(stacks)

    def rc_msg(flat, off, nh=None, n=None):
        n = len(off) - 1 if n is None else n
        f = np.ascontiguousarray(flat, dtype=scb200.MOVE_DTYPE)
        o = np.ascontiguousarray(off, dtype=np.int32)
        h = None if nh is None else np.ascontiguousarray(nh, dtype=np.int8)
        bufs = [np.zeros((max(n, 1), scb200.SC_MAX_MOVES), np.uint32), np.zeros(max(n, 1), np.int32),
                np.zeros((max(n, 1), scb200.SC_MAX_MOVES), np.float32), np.zeros(max(n, 1), np.float32)]
        rc = L.sc_predict_stack(e.handle, n, f.ctypes.data if len(f) else None, o.ctypes.data,
                                None if h is None else h.ctypes.data, None, *(b.ctypes.data for b in bufs), None)
        return rc, L.sc_last_error().decode()

    assert rc_msg(flat, off)[0] == 0
    o2 = off.copy()
    o2 += 1
    rc, msg = rc_msg(flat, o2)
    assert rc == -1 and "stack_off[0]" in msg
    o2 = off.copy()
    o2[3] = o2[2] - 1
    rc, msg = rc_msg(flat, o2)
    assert rc == -1 and "decreases at leaf 2" in msg
    long = [(12, 28, 0)] * (scb200.SC_MAX_STACK + 1)
    rc, msg = rc_msg(*_flat([[], long]))
    assert rc == -1 and "leaf 1" in msg and "SC_MAX_STACK" in msg
    for field, value in (("from", 64), ("to", 64), ("from", 255), ("promo", 1), ("promo", 6)):
        f2 = flat.copy()
        f2[field][5] = value
        rc, msg = rc_msg(f2, off)
        assert rc == -1 and "stack[5]" in msg, (field, value)
    lens = np.diff(off)
    for leaf, value in ((2, 0), (2, 9), (2, -1)):
        nh = np.minimum(lens + 1, 8).astype(np.int8)
        nh[leaf] = value
        rc, msg = rc_msg(flat, off, nh)
        assert rc == -1 and f"n_hist[{leaf}]" in msg, (leaf, value)
    # more history slots than the stack has positions
    rc, msg = rc_msg(*_flat([[]]), nh=[2])
    assert rc == -1 and "n_hist[0]" in msg
    rc, msg = rc_msg(*_flat([[], _uci("e2e4 e7e5")]), nh=[1, 4])
    assert rc == -1 and "n_hist[1]" in msg
    assert rc_msg(*_flat([[], _uci("e2e4 e7e5")]), nh=[1, 3])[0] == 0
    # n > max_batch, NULL offsets
    f9, o9 = _flat(random_leaves.stacks[:9])
    assert e.predict_stack((f9, o9), check=False)[0] == -1
    with pytest.raises(scb200.SCError):
        e.predict_stack((f9, o9))
    z = np.zeros(4, np.float32)
    assert L.sc_predict_stack(e.handle, 1, None, None, None, None, z.ctypes.data, z.ctypes.data, z.ctypes.data,
                              z.ctypes.data, None) == -1
    # n = 0 returns at once; an empty stack is the start position
    assert L.sc_predict_stack(e.handle, 0, None, None, None, None, None, None, None, None, None) == 0
    assert e.predict_stack([])[1].shape == (0,)
    _, cnt, _, _, pos = e.predict_stack([[]], positions=True)
    start = scb200.rules_probe([])[1]
    assert cnt[0] == 20 and pos[0].tobytes() == np.array([start], dtype=scb200.POSITION_DTYPE)[0].tobytes()
    moves, cnt, _, _ = e.predict_stack(stacks)
    assert cnt.tolist() == [len(m) for m in random_leaves.moves[100:108]]
    e.close()


def _rejections():
    """One stack per replay-time rejection: (stack, rejected ply, words the message must hold)."""
    pawn_on_h7 = _uci("h2h4 g7g5 h4g5 h7h6 g5h6 g8f6 h6h7 a7a6")
    return [
        (_uci("e2e4 e2e4"), 1, "from-square holds no piece of the side to move"),    # e2 is empty
        (_uci("e2e4 e4e5"), 1, "from-square holds no piece of the side to move"),    # Black to move, e4 is White's
        (_uci("g1f3 g8f6 f3h2"), 2, "to-square holds a piece of the side to move"),  # own pawn on h2
        ([(0, 60, 0)], 0, "or a king"),                                               # Ra1 onto the black king
        (_uci("g1f3") + [(62, 45, 5)], 1, "promotes a piece that is not a pawn"),     # Ng8-f6=Q
        (_uci("e2e4") + [(52, 44, 2)], 1, "promotes a piece that is not a pawn"),     # e7-e6=N
        (pawn_on_h7 + [(55, 63, 0)], 8, "without a promotion"),                       # hxh8 naming no piece
    ]


def test_replay_rejections(engine):
    import scb200

    L = scb200.load_library()
    for stack, ply, words in _rejections():
        # alone, and as leaf 2 of 3
        for stacks, leaf in (([stack], 0), ([[], _uci("d2d4"), stack], 2)):
            flat, off = _flat(stacks)
            rc, pos, moves, cnt, _ = _raw_predict_stack(engine, flat, off)
            msg = L.sc_last_error().decode()
            assert rc == -1 and f"leaf {leaf}, ply {ply}" in msg and words in msg, (stack, msg)
            # the leaf is packed from the moves before the rejected one
            exp = _expected(np.array([scb200.rules_probe(stack[:ply])[1]], dtype=scb200.POSITION_DTYPE), [min(8, ply + 1)])
            _assert_packed_equal(pos[leaf : leaf + 1], exp, [stack[:ply]])
            if leaf:  # the real leaves next to it: the start position and 1.d4
                assert cnt[:2].tolist() == [20, len(scb200.rules_probe(_uci("d2d4"))[0])]


def test_garbage_stacks_stay_in_their_slots(engine, random_leaves):
    import scb200

    rng = np.random.RandomState(23)
    n = 1024
    stacks = []
    for i in range(n):
        if i % 2 == 0:
            stacks.append(random_leaves.stacks[3 * i])
        else:
            ln = rng.randint(0, 300)
            stacks.append(list(zip(rng.randint(0, 64, ln), rng.randint(0, 64, ln), rng.choice([0, 2, 3, 4, 5], ln))))
    flat, off = _flat(stacks)
    for batch in ((flat, off), _flat(stacks[:40])):  # device buffers, and the pinned staging buffer
        m = len(batch[1]) - 1
        rc, pos, moves, cnt, _ = _raw_predict_stack(engine, *batch, guard_rows=3)
        assert rc in (0, -1)
        assert ((cnt >= 0) & (cnt <= scb200.SC_MAX_MOVES)).all()
        host, _ = random_leaves.positions(slice(None))
        for i in range(0, m, 2):
            j = 3 * i
            exp = _expected(host[j : j + 1], [min(8, len(stacks[i]) + 1)])
            _assert_packed_equal(pos[i : i + 1], exp, stacks[i : i + 1])
            got = [tuple(int(x) for x in (r["from"], r["to"], r["promo"])) for r in moves[i, : cnt[i]]]
            assert got == random_leaves.moves[j], i
    # the engine answers a normal call afterwards
    _, c, _, _ = engine.predict_stack(random_leaves.stacks[:4])
    assert c.tolist() == [len(x) for x in random_leaves.moves[:4]]
