"""sc_predict: `Game::predict` with the legal moves generated on the device.

The device runs the host driver's generator (csrc/host/chess_rules.hpp, pinned to python-chess by the perft tables, the
C oracle and the sample games), so its moves must equal the host's in number and order.  Priors and values come from the
same network and the same gather as sc_eval, so they must equal sc_eval's bit for bit when sc_eval is given the host's
moves.  A terminal leaf (no legal moves) gets torch.rs:98-106's value.
"""
import ast
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ("SC_MODE_FP32", "SC_MODE_BF16", "SC_MODE_FP32_FFMA", "SC_MODE_FP16")
PERFT_FENS = [  # the six positions of tests/test_search_host.py::test_native_rules_perft_matches_published_tables
    "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1",
    "8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1",
    "r3k2r/Pppp1ppp/1b3nbN/nP6/BBP1P3/q4N2/Pp1P2PP/R2Q1RK1 w kq - 0 1",
    "rnbq1k1r/pp1Pbppp/2p5/8/2B5/8/PPP1NnPP/RNBQK2R w KQ - 1 8",
    "r4rk1/1pp1qppp/p1np1n2/2b1p1B1/2B1P1b1/P1NP1N2/1PP1QPPP/R4RK1 w - - 0 10",
    "1k1r4/1r5p/p4n1P/1ppP1P2/PP6/4PP1b/3B4/R1N1K3 b - - 0 39",
]
MOVES_218 = "R6R/3Q4/1Q4Q1/4Q3/2Q4Q/Q4Q2/pp1Q4/kBNN1KB1 w - - 0 1"
TERMINAL_FENS = [  # (fen, value in White's perspective)
    ("rnb1kbnr/pppp1ppp/8/4p3/6Pq/5P2/PPPPP2P/RNBQKBNR w KQkq - 1 3", -1.0),  # fool's mate: White is mated
    ("6rk/5Npp/8/8/8/8/8/6K1 b - - 0 1", 1.0),                               # smothered mate: Black is mated
    ("7k/5Q2/6K1/8/8/8/8/8 b - - 0 1", 0.0),                                 # stalemate
    ("8/8/8/8/8/5k2/5p2/5K2 w - - 0 1", 0.0),                                # stalemate, bare pawn ending
]


def _edge_fens():
    """EDGE_FENS of oracle/make_golden_pychess.py, read without importing it (it needs python-chess)."""
    with open(os.path.join(ROOT, "oracle", "make_golden_pychess.py")) as f:
        tree = ast.parse(f.read())
    for node in tree.body:
        if isinstance(node, ast.Assign) and node.targets[0].id == "EDGE_FENS":
            return ast.literal_eval(node.value)
    raise AssertionError("EDGE_FENS not found")


def _fen_ep(fen):
    f = fen.split()[3]
    return -1 if f == "-" else (int(f[1]) - 1) * 8 + ord(f[0]) - ord("a")


class Leaves:
    """Positions with the host generator's answer: packed leaf, python-chess ep_square, legal moves, terminal value."""

    def __init__(self):
        self.pos, self.ep, self.moves, self.value = [], [], [], []

    def add(self, hist, fen=None):
        import scb200

        mv, pos, (term, _) = scb200.rules_probe(hist, fen)
        if hist:
            f, t, _ = hist[-1]
            pawn = (int(pos["slot"][0][0]) >> t) & 1
            ep = (f + t) // 2 if pawn and abs(t - f) == 16 else -1
        else:
            ep = _fen_ep(fen) if fen else -1
        self.pos.append(pos)
        self.ep.append(ep)
        self.moves.append([tuple(int(x) for x in m) for m in mv])
        # no legal moves: outcome() names checkmate first, every other termination is a draw for `predict`
        self.value.append((-1.0 if pos["meta"][0] else 1.0) if term == 1 else 0.0)
        return mv

    def arrays(self, sl=slice(None)):
        import scb200

        pos = np.array(self.pos[sl], dtype=scb200.POSITION_DTYPE)
        return pos, np.array(self.ep[sl], dtype=np.int8)

    def csr(self, sl=slice(None)):
        import scb200

        mv = self.moves[sl]
        off = np.zeros(len(mv) + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(m) for m in mv])
        flat = np.zeros(max(1, int(off[-1])), dtype=scb200.MOVE_DTYPE)
        k = 0
        for ms in mv:
            for m in ms:
                flat[k] = (m[0], m[1], m[2], 0)
                k += 1
        return flat, off


def _random_play(leaves, n, seed):
    """Seeded uniform random play with the host generator until n positions (terminal ones included) are recorded."""
    rng = np.random.RandomState(seed)
    while len(leaves.pos) < n:
        hist = []
        for _ in range(200):
            mv = leaves.add(hist)
            if len(mv) == 0 or len(leaves.pos) >= n:
                break
            hist.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))


@pytest.fixture(scope="module")
def blob(tmp_path_factory):
    import net
    import scb200

    p = str(tmp_path_factory.mktemp("predict") / "w.scw")
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
    lv = Leaves()
    _random_play(lv, 20000, seed=11)
    return lv


def _check_moves(engine, lv):
    n_all = len(lv.pos)
    for b in range(0, n_all, engine.max_batch):
        sl = slice(b, min(n_all, b + engine.max_batch))
        pos, ep = lv.arrays(sl)
        moves, cnt, _, val = engine.predict(pos, ep)
        for i, exp in enumerate(lv.moves[sl]):
            assert cnt[i] == len(exp), (b + i, cnt[i], len(exp))
            got = [(int(m["from"]), int(m["to"]), int(m["promo"])) for m in moves[i, : cnt[i]]]
            assert got == exp, b + i
            if not exp:
                assert val[i] == lv.value[b + i], (b + i, val[i])
    return n_all


def test_moves_match_host_generator_on_sample_games(engine, sample_games):
    lv = Leaves()
    for game in sample_games["games"]:
        hist = []
        ucis = game["uci"].split()
        for ply in range(len(ucis) + 1):
            lv.add(hist)
            if ply < len(ucis):
                u = ucis[ply]
                sq = lambda s: (int(s[1]) - 1) * 8 + ord(s[0]) - ord("a")  # noqa: E731
                hist.append((sq(u[:2]), sq(u[2:4]), " pnbrqk".index(u[4]) if len(u) > 4 else 0))
    assert _check_moves(engine, lv) > 3500


def test_moves_match_host_generator_on_edge_fens_and_continuations(engine):
    lv = Leaves()
    rng = np.random.RandomState(3)
    for fen in _edge_fens() + [MOVES_218] + [f for f, _ in TERMINAL_FENS]:
        for _ in range(3):
            hist = []
            for _ in range(40):
                mv = lv.add(hist, fen)
                if len(mv) == 0:
                    break
                hist.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
    assert max(len(m) for m in lv.moves) == 218
    _check_moves(engine, lv)


def test_moves_match_host_generator_on_random_play(engine, random_leaves):
    lv = random_leaves
    # ep_square comes from the last move: every kind of leaf is there
    assert sum(e >= 0 for e in lv.ep) > 200 and sum(len(m) == 0 for m in lv.moves) > 10
    assert _check_moves(engine, lv) == 20000


def test_moves_match_host_generator_within_two_plies_of_perft_positions(engine):
    lv = Leaves()
    for fen in PERFT_FENS:
        for m1 in lv.add([], fen):
            h1 = [tuple(int(x) for x in m1)]
            for m2 in lv.add(h1, fen):
                lv.add(h1 + [tuple(int(x) for x in m2)], fen)
    assert len(lv.pos) > 6500
    _check_moves(engine, lv)


def test_terminal_leaves(engine):
    import scb200

    lv = Leaves()
    for fen, _ in TERMINAL_FENS:
        lv.add([], fen)
    pos, ep = lv.arrays()
    moves, cnt, _, val = engine.predict(pos, ep)
    assert cnt.tolist() == [0] * len(TERMINAL_FENS)
    assert val.tolist() == [v for _, v in TERMINAL_FENS]
    # in a batch with non-terminal leaves, and on the latency path (one leaf)
    for i, (fen, v) in enumerate(TERMINAL_FENS):
        m1, c1, _, v1 = engine.predict(pos[i : i + 1], ep[i : i + 1])
        assert c1[0] == 0 and v1[0] == v
    start = scb200.rules_probe([])[1]
    mix = np.array([start, pos[0], start, pos[2]], dtype=scb200.POSITION_DTYPE)
    _, c, _, v = engine.predict(mix)
    assert c.tolist() == [20, 0, 20, 0] and v[1] == -1.0 and v[3] == 0.0


@pytest.mark.parametrize("mode", MODES)
def test_priors_and_values_equal_sc_eval(blob, random_leaves, mode):
    """n = 1 / 37 (pinned staging; bf16/fp16: latency kernel), 129 (device buffers) and 2048 (throughput kernel)."""
    import scb200

    e = scb200.Engine(blob, 0, getattr(scb200, mode), 2048)
    lv = random_leaves
    for n in (1, 37, 129, 2048):
        for start in (0, 5000):
            sl = slice(start, start + n)
            pos, ep = lv.arrays(sl)
            moves, off = lv.csr(sl)
            pe, ve = e.eval(pos, moves, off)
            mp, cnt, pp, vp = e.predict(pos, ep)
            assert np.array_equal(cnt, np.diff(off)), (mode, n)
            for i in range(n):
                c = int(cnt[i])
                assert np.array_equal(pp[i, :c].view(np.uint32), pe[off[i] : off[i + 1]].view(np.uint32)), (mode, n, i)
                exp_v = ve[i] if c else lv.value[start + i]
                assert np.float32(vp[i]).view(np.uint32) == np.float32(exp_v).view(np.uint32), (mode, n, i)
    # the policy gather of the predict leg sees exactly the moves it would see in sc_eval: a second call agrees
    pos, ep = lv.arrays(slice(0, 37))
    a, b = e.predict(pos, ep), e.predict(pos, ep)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
    e.close()


def _raw_predict(engine, pos, ep, guard_rows=1):
    """sc_predict through ctypes with one guard row past the n output rows, to see every byte the call writes."""
    import scb200

    n = len(pos)
    moves = np.full((n + guard_rows, scb200.SC_MAX_MOVES), 0xAB, dtype=np.uint32)
    cnt = np.full(n + guard_rows, -7, dtype=np.int32)
    priors = np.full((n + guard_rows, scb200.SC_MAX_MOVES), 7.0, dtype=np.float32)
    vals = np.full(n + guard_rows, 7.0, dtype=np.float32)
    pos = np.ascontiguousarray(pos, dtype=scb200.POSITION_DTYPE)
    ep = None if ep is None else np.ascontiguousarray(ep, dtype=np.int8)
    rc = scb200.load_library().sc_predict(engine.handle, n, pos.ctypes.data, None if ep is None else ep.ctypes.data,
                                          moves.ctypes.data, cnt.ctypes.data, priors.ctypes.data, vals.ctypes.data, None)
    assert (moves[n:] == 0xAB).all() and (cnt[n:] == -7).all() and (priors[n:] == 7.0).all() and (vals[n:] == 7.0).all()
    return rc, moves[:n].view(scb200.MOVE_DTYPE), cnt[:n], priors[:n], vals[:n]


# a position without kings whose side to move has 261 pseudo-legal (and, without a king, legal) moves: 18 queens, a bishop
OVERFLOW_BOARDS = [0, 0, 0x0100000000000000, 0, 0xEE114141414210EF, 0]


def test_garbage_positions_stay_in_their_slots(engine, random_leaves):
    import scb200

    rng = np.random.RandomState(9)
    n = 1024
    raw = rng.randint(0, 256, size=n * scb200.POSITION_DTYPE.itemsize, dtype=np.uint8)
    pos = raw.view(scb200.POSITION_DTYPE).copy()
    for k in range(1, 4):  # sparser boards too: more sliders with open lines
        sl = slice(k, None, 4)
        pos["slot"][sl] &= rng.randint(0, 2**63, size=pos["slot"][sl].shape, dtype=np.int64).astype(np.uint64) << np.uint64(1)
    ep = rng.choice([-1] + list(range(16, 24)) + list(range(40, 48)), size=n).astype(np.int8)
    # every other leaf is a real one: a generator that wrote past its slot would corrupt its neighbour's moves
    real_pos, real_ep = random_leaves.arrays(slice(0, n // 2))
    pos[0::2], ep[0::2] = real_pos, real_ep
    rc, moves, cnt, _, _ = _raw_predict(engine, pos, ep)
    assert rc in (0, -1)
    assert ((cnt >= 0) & (cnt <= scb200.SC_MAX_MOVES)).all()
    for i in range(0, n, 2):
        exp = random_leaves.moves[i // 2]
        assert cnt[i] == len(exp) and [tuple(int(x) for x in (m["from"], m["to"], m["promo"])) for m in moves[i, : cnt[i]]] == exp
    # more pseudo-legal moves than a slot holds: SC_E_INVAL, at most SC_MAX_MOVES written, the neighbours intact
    bad = np.zeros(1, dtype=scb200.POSITION_DTYPE)
    for k, b in enumerate(OVERFLOW_BOARDS):
        bad["slot"][0, 0, k] = b
    bad["slot"][0, 0, 6] = sum(OVERFLOW_BOARDS)
    bad["meta"][0] = (1, 1, 0, 0, 0, 0, 0)
    bad["n_hist"][0] = 1
    trio = np.concatenate([real_pos[:1], bad, real_pos[1:2]])
    for batch in (trio, np.concatenate([trio] * 60)):  # staging buffers, and device buffers
        rc, moves, cnt, _, _ = _raw_predict(engine, batch, None)
        assert rc == -1 and "pseudo-legal" in scb200.load_library().sc_last_error().decode()
        assert cnt[1] == scb200.SC_MAX_MOVES
        assert cnt[0] == len(random_leaves.moves[0]) and cnt[2] == len(random_leaves.moves[1])
    # the engine is fine afterwards
    m, c, _, _ = engine.predict(real_pos[:4], real_ep[:4])
    assert c.tolist() == [len(x) for x in random_leaves.moves[:4]]


def test_bad_arguments(blob, random_leaves):
    import scb200

    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 8)
    pos, ep = random_leaves.arrays(slice(0, 8))
    for bad in (-2, 0, 7, 15, 24, 39, 48, 63, 127, -128):
        e2 = ep.copy()
        e2[5] = bad
        rc = e.predict(pos, e2, check=False)[0]
        assert rc == -1 and "ep_square[5]" in scb200.load_library().sc_last_error().decode(), bad
    pos9 = np.concatenate([pos, pos[:1]])
    assert e.predict(pos9, check=False)[0] == -1
    with pytest.raises(scb200.SCError):
        e.predict(pos9)
    assert e.predict(pos[:0])[1].shape == (0,)
    moves, cnt, _, _ = e.predict(pos, ep)
    assert cnt.tolist() == [len(m) for m in random_leaves.moves[:8]]
    e.close()
