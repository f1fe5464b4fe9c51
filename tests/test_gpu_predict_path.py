"""sc_set_roots / sc_predict_path: leaves given as a stored root game plus the moves played after it.

The contract is bit-identity to sc_predict_stack on the concatenated stack root ++ path: packed leaves, moves, counts,
priors, values, terminal rule, status codes and the plies in messages.  So sc_predict_stack (itself checked against
the host rules in test_gpu_predict_stack.py) is the oracle of every test here.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ("SC_MODE_FP32", "SC_MODE_BF16", "SC_MODE_FP32_FFMA", "SC_MODE_FP16")
SC_E_INVAL, SC_E_STATE = -1, -5


def _sq(s):
    return (int(s[1]) - 1) * 8 + ord(s[0]) - ord("a")


def _uci(text):
    return [(_sq(u[:2]), _sq(u[2:4]), " pnbrqk".index(u[4]) if len(u) > 4 else 0) for u in text.split()]


KNIGHTS = _uci("g1f3 g8f6 f3g1 f6g8")  # back to the start position every four plies


def _rook_shuffle_300():
    """300 reversible plies of rook moves after the opening pawn moves: the halfmove clock passes 150"""
    rooks = _uci("a2a4 a7a5 a1a3 a8a6")
    w, b = 0, 0
    for k in range(300):
        if k % 2 == 0:
            rooks.append((16 + w, 16 + (w + 1) % 8, 0))  # a3 .. h3 and round
            w = (w + 1) % 8
        else:
            rooks.append((40 + b, 40 + (b + 1) % 7, 0))  # a6 .. g6 and round
            b = (b + 1) % 7
    return rooks


# move lists whose repetition flags, castling rights and en-passant keys the packing depends on; every split of each
# into root and path is checked
BOUNDARY_SEQUENCES = {
    # 2-, 3- and 5-fold repetitions of the start position at plies 4, 8 and 16
    "shuffle_5fold": KNIGHTS * 4 + _uci("g1f3"),
    # the white king and a rook lose their castling rights early; the shuffles that follow repeat without them
    "king_move": _uci("e2e4 e7e5") + KNIGHTS * 2 + _uci("e1e2 e8e7 e2e1 e7e8") * 3,
    "rook_move": _uci("g1f3 g8f6 h1g1 h8g8 g1h1 g8h8") + _uci("b1c3 b8c6 c3b1 c6b8") * 3,
    # the bishop takes the rook on h8: Black loses its kingside right without moving the rook
    "rook_captured": _uci("b2b3 g7g5 c1b2 g8h6 b2h8") + _uci("b8c6 b1c3 c6b8 c3b1") * 3,
    # d7d5 is the root's last move and exd6 (legal) the path's first; the key after d7d5 carries the ep square
    "ep_legal": _uci("e2e4 a7a6 e4e5 d7d5 e5d6") + _uci("g8f6 g1f3 f6g8 f3g1") * 2,
    "ep_legal_declined": _uci("e2e4 a7a6 e4e5 d7d5") + _uci("g1f3 g8f6 f3g1 f6g8") * 2,
    # e2e4 is the root's last move; dxe3 is only pseudo-legal (the d4 pawn is pinned by Bb2 against Kf6)
    "ep_pinned": _uci("b2b3 d7d5 c1b2 d5d4 b1a3 f7f5 a3b1 e8f7 b1a3 f7f6 e2e4 d4e3"),
    "ep_pinned_declined": _uci("b2b3 d7d5 c1b2 d5d4 b1a3 f7f5 a3b1 e8f7 b1a3 f7f6 e2e4")
    + _uci("f6f7 a3b1 f7f6 b1a3") * 2,
}


def _random_games(n_games, max_plies, seed):
    """seeded uniform random games of up to max_plies plies (they end early at mate or stalemate)"""
    import scb200

    rng = np.random.RandomState(seed)
    games = []
    for _ in range(n_games):
        hist = []
        while len(hist) < max_plies:
            mv = scb200.rules_probe(hist)[0]
            if len(mv) == 0:
                break
            hist.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
        games.append(hist)
    return games


def _assert_same(got, exp, what):
    """predict_path's outputs (moves, counts, priors, values, positions) against predict_stack's, bit for bit"""
    moves, cnt, priors, vals, pos = got
    emoves, ecnt, epriors, evals, epos = exp
    assert np.array_equal(cnt, ecnt), what
    for i in range(len(cnt)):
        c = int(cnt[i])
        assert np.array_equal(moves[i, :c].view(np.uint32), emoves[i, :c].view(np.uint32)), (what, i)
        assert np.array_equal(priors[i, :c].view(np.uint32), epriors[i, :c].view(np.uint32)), (what, i)
        assert pos[i].tobytes() == epos[i].tobytes(), (what, i)
    assert np.array_equal(vals.view(np.uint32), evals.view(np.uint32)), what


def _check_against_stack(e, roots, leaf_root, paths, n_hist=None, what="", set_roots=True):
    """sets `roots` (unless set_roots is False) and checks predict_path on every leaf against predict_stack on
    root ++ path, in batches of the engine's max_batch; returns the number of leaves"""
    if set_roots:
        e.set_roots(roots)
    for b in range(0, len(paths), e.max_batch):
        sl = slice(b, b + e.max_batch)
        lr, ps = list(leaf_root[sl]), list(paths[sl])
        nh = None if n_hist is None else n_hist[sl]
        got = e.predict_path(lr, ps, n_hist=nh, positions=True)
        exp = e.predict_stack([list(roots[r]) + list(p) for r, p in zip(lr, ps)], n_hist=nh, positions=True)
        _assert_same(got, exp, (what, b))
    return len(paths)


@pytest.fixture(scope="module")
def blob(tmp_path_factory):
    import net
    import scb200

    p = str(tmp_path_factory.mktemp("predict_path") / "w.scw")
    scb200.write_blob(net.perturb_norm_params(net.init_state_dict(2, 7), 1234), p)
    return p


@pytest.fixture(scope="module")
def engine(blob):
    import scb200

    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 2048)
    yield e
    e.close()


@pytest.fixture(scope="module")
def random_games():
    """48 seeded random-play games of up to 300 plies"""
    games = _random_games(48, 300, seed=11)
    assert max(len(g) for g in games) == 300
    return games


def _leaf_batch(games, n, n_roots, rng):
    """n leaves over n_roots roots (prefixes of `games` of random length), in shuffled root order, paths 0..30 plies
    continuing each root's game; with more than one root, root 1 is the empty game"""
    roots, root_game = [], []
    for r in range(n_roots):
        g = games[r % len(games)]
        a = 0 if r == 1 else rng.randint(0, len(g) + 1)
        roots.append(g[:a])
        root_game.append(g)
    leaf_root = rng.permutation(np.arange(n) % n_roots)
    paths = []
    for r in leaf_root:
        a, g = len(roots[r]), root_game[r]
        paths.append(g[a : a + rng.randint(0, min(30, len(g) - a) + 1)])
    return roots, leaf_root, paths


@pytest.mark.parametrize("mode", MODES)
def test_outputs_equal_predict_stack(blob, random_games, mode):
    """n = 1 / 37 (pinned staging; bf16/fp16: latency kernel), 129 (device buffers) and 2048 (throughput kernel); one
    root per leaf and 16 roots shared by many leaves"""
    import scb200

    e = scb200.Engine(blob, 0, getattr(scb200, mode), 2048)
    rng = np.random.RandomState(3)
    for n in (1, 37, 129, 2048):
        for n_roots in sorted({n, min(n, 16)}):
            roots, leaf_root, paths = _leaf_batch(random_games, n, n_roots, rng)
            _check_against_stack(e, roots, leaf_root, paths, what=(mode, n, n_roots))
    e.close()


def test_sample_game_roots(engine, sample_games):
    """roots at every fourth ply of every sample game, each shared by four leaves whose paths (0..30 plies) follow the
    game, and one root shared by 300 leaves along random continuations (siblings of one search)"""
    import scb200

    rng = np.random.RandomState(7)
    roots, index, leaf_root, paths = [], {}, [], []
    for gi, game in enumerate(sample_games["games"]):
        g = _uci(game["uci"])
        for a in range(0, len(g) + 1, 4):
            index[(gi, a)] = len(roots)
            roots.append(g[:a])
        for a in range(0, len(g) + 1, 4):
            for _ in range(4):
                leaf_root.append(index[(gi, a)])
                paths.append(g[a : a + rng.randint(0, min(30, len(g) - a) + 1)])
    assert len(roots) <= engine.max_batch
    assert _check_against_stack(engine, roots, leaf_root, paths, what="sample") > 2000
    # one root, many siblings: random legal continuations of 0..12 plies from the same position
    g = _uci(sample_games["games"][3]["uci"])
    root = g[:40]
    paths = []
    for _ in range(300):
        p = []
        for _ in range(rng.randint(0, 13)):
            mv = scb200.rules_probe(root + p)[0]
            if len(mv) == 0:
                break
            p.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
        paths.append(p)
    _check_against_stack(engine, [root], [0] * len(paths), paths, what="siblings")


def test_every_n_hist(engine, random_games):
    """every n_hist 1..8 with paths of 0..7 plies after roots of 0..12 and of random length: the history slots reach
    back into the root's records, and for short games to the initial position"""
    rng = np.random.RandomState(9)
    roots, leaf_root, paths, n_hist = [], [], [], []
    for g in [g for g in random_games if len(g) >= 40][:24]:
        for a in list(range(0, 13)) + [int(rng.randint(13, len(g) - 7))]:
            r = len(roots)
            roots.append(g[:a])
            for ln in range(0, 8):
                for h in range(1, min(8, a + ln + 1) + 1):
                    leaf_root.append(r)
                    paths.append(g[a : a + ln])
                    n_hist.append(h)
    n_hist = np.array(n_hist, dtype=np.int8)
    assert _check_against_stack(engine, roots, leaf_root, paths, n_hist=n_hist, what="n_hist") > 5000


@pytest.mark.parametrize("name", sorted(BOUNDARY_SEQUENCES))
def test_boundary_sequences_at_every_split(engine, name):
    """every (root, path) split of a built sequence: repetitions that start in the root and complete in the path,
    castling rights lost in the root, en passant (legal and pinned) as the path's first move after a double push as
    the root's last, and the empty path"""
    seq = BOUNDARY_SEQUENCES[name]
    roots = [seq[:a] for a in range(len(seq) + 1)]
    leaf_root, paths = [], []
    for a in range(len(seq) + 1):
        for b in range(a, min(len(seq), a + 30) + 1):
            leaf_root.append(a)
            paths.append(seq[a:b])
    _check_against_stack(engine, roots, leaf_root, paths, what=name)
    if name == "shuffle_5fold":  # the 2-, 3- and 5-fold repetitions are in the packed flags
        _, _, _, _, pos = engine.predict_path([0, 0, 4], [seq[:4], seq[:8], seq[4:16]], positions=True)
        assert [int(p["slot"][0][7]) for p in pos] == [1, 3, 3]


def test_reversible_stretch_split(engine):
    """300 reversible plies split at several points, past the 75-move clock: repetition walks and the halfmove run
    cross the root / path boundary"""
    seq = _rook_shuffle_300()
    cuts = (0, 3, 4, 5, 60, 149, 150, 151, 152, 153, 200, 274, 290, len(seq))
    leaf_root, paths = [], []
    for r, a in enumerate(cuts):
        for ln in range(0, min(30, len(seq) - a) + 1):
            leaf_root.append(r)
            paths.append(seq[a : a + ln])
    _check_against_stack(engine, [seq[:a] for a in cuts], leaf_root, paths, what="rook_shuffle")
    _, _, _, _, pos = engine.predict_path([len(cuts) - 1], [[]], positions=True)
    assert int(pos[0]["meta"][6]) > 150


def test_empty_path_equals_root_alone(engine, random_games):
    import scb200

    roots = [g[: 37 * (i % 9)] for i, g in enumerate(random_games)]
    engine.set_roots(roots)
    got = engine.predict_path(np.arange(len(roots)), [[]] * len(roots), positions=True)
    exp = engine.predict_stack(roots, positions=True)
    _assert_same(got, exp, "empty path")
    # the start position
    engine.set_roots([[]])
    got = engine.predict_path([0], [[]], positions=True)
    start = scb200.rules_probe([])[1]
    assert got[1][0] == 20 and got[4][0].tobytes() == np.array([start], dtype=scb200.POSITION_DTYPE)[0].tobytes()


def _flat(lists):
    import scb200

    off = np.zeros(len(lists) + 1, dtype=np.int32)
    off[1:] = np.cumsum([len(s) for s in lists])
    flat = np.zeros(int(off[-1]), dtype=scb200.MOVE_DTYPE)
    for s, o in zip(lists, off[:-1]):
        for k, m in enumerate(s):
            flat[o + k] = (m[0], m[1], m[2], 0)
    return flat, off


def _raw_set_roots(e, roots):
    import scb200

    flat, off = _flat(roots)
    rc = scb200.load_library().sc_set_roots(e.handle, len(roots), flat.ctypes.data if len(flat) else None,
                                            off.ctypes.data)
    return rc, scb200.load_library().sc_last_error().decode()


def _raw_predict_path(e, root, flat, off, n_hist=None, guard_rows=1):
    """sc_predict_path through ctypes with guard rows past the n output rows, to see every byte the call writes"""
    import scb200

    n = len(off) - 1
    rows = n + guard_rows
    pos = np.full(rows, 0x5A, dtype=np.uint8).repeat(scb200.POSITION_DTYPE.itemsize).view(scb200.POSITION_DTYPE).copy()
    moves = np.full((rows, scb200.SC_MAX_MOVES), 0xAB, dtype=np.uint32)
    cnt = np.full(rows, -7, dtype=np.int32)
    priors = np.full((rows, scb200.SC_MAX_MOVES), 7.0, dtype=np.float32)
    vals = np.full(rows, 7.0, dtype=np.float32)
    root = np.ascontiguousarray(root, dtype=np.int32)
    flat = np.ascontiguousarray(flat, dtype=scb200.MOVE_DTYPE)
    off = np.ascontiguousarray(off, dtype=np.int32)
    nh = None if n_hist is None else np.ascontiguousarray(n_hist, dtype=np.int8)
    L = scb200.load_library()
    rc = L.sc_predict_path(e.handle, n, root.ctypes.data if n else None, flat.ctypes.data if len(flat) else None,
                           off.ctypes.data, None if nh is None else nh.ctypes.data, pos.ctypes.data, moves.ctypes.data,
                           cnt.ctypes.data, priors.ctypes.data, vals.ctypes.data, None)
    msg = L.sc_last_error().decode()
    assert (pos[n:].view(np.uint8) == 0x5A).all()
    assert (moves[n:] == 0xAB).all() and (cnt[n:] == -7).all() and (priors[n:] == 7.0).all() and (vals[n:] == 7.0).all()
    return rc, msg, (moves[:n].view(scb200.MOVE_DTYPE), cnt[:n], priors[:n], vals[:n], pos[:n])


def _rejections():
    """(stack, rejected ply, words the message must hold), one per replay-time rejection"""
    pawn_on_h7 = _uci("h2h4 g7g5 h4g5 h7h6 g5h6 g8f6 h6h7 a7a6")
    return [
        (_uci("e2e4 e2e4"), 1, "from-square holds no piece of the side to move"),
        (_uci("g1f3 g8f6 f3h2"), 2, "to-square holds a piece of the side to move"),
        (_uci("e2e4 e7e5") + [(3, 60, 0)], 2, "or a king"),
        (_uci("g1f3") + [(62, 45, 5)], 1, "promotes a piece that is not a pawn"),
        (pawn_on_h7 + [(55, 63, 0)], 8, "without a promotion"),
    ]


def test_state_errors(blob, random_games):
    import scb200

    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 64)
    flat, off = _flat([random_games[0][:3]])
    # before any sc_set_roots, also for n = 0
    assert _raw_predict_path(e, [0], flat, off)[0] == SC_E_STATE
    assert scb200.load_library().sc_predict_path(e.handle, 0, None, None, None, None, None, None, None, None, None,
                                                 None) == SC_E_STATE
    with pytest.raises(scb200.SCError, match="no roots"):
        e.predict_path([0], [[]])
    e.set_roots([random_games[0][:10]])
    assert _raw_predict_path(e, [0], *_flat([random_games[0][10:13]]))[0] == 0
    # a root rejected at replay time: the message names the root and the ply, and the engine is left without roots
    for stack, ply, words in _rejections():
        rc, msg = _raw_set_roots(e, [[], random_games[1][:20], stack])
        assert rc == SC_E_INVAL and f"sc_set_roots: root 2, ply {ply}" in msg and words in msg, msg
        assert _raw_predict_path(e, [0], *_flat([[]]))[0] == SC_E_STATE
        e.set_roots([[]])
    # n_roots = 0 clears the table
    e.set_roots([])
    assert _raw_predict_path(e, [0], *_flat([[]]))[0] == SC_E_STATE
    e.close()


def test_argument_errors(blob, random_games):
    import scb200

    L = scb200.load_library()
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 8)
    g = max(random_games, key=len)
    roots = [g[:5], g[:40], g[:41]]
    e.set_roots(roots)
    paths = [g[5:9], g[40:41], []]
    flat, off = _flat(paths)
    assert _raw_predict_path(e, [0, 1, 2], flat, off)[0] == 0
    for bad in (-1, 3, 1 << 30):
        rc, msg, _ = _raw_predict_path(e, [0, bad, 2], flat, off)
        assert rc == SC_E_INVAL and f"root[1] = {bad} is not in 0..2" in msg, msg
    o2 = off + 1
    rc, msg, _ = _raw_predict_path(e, [0, 1, 2], flat, o2)
    assert rc == SC_E_INVAL and "path_off[0]" in msg
    o2 = off.copy()
    o2[2] = o2[1] - 1
    rc, msg, _ = _raw_predict_path(e, [0, 1, 2], flat, o2)
    assert rc == SC_E_INVAL and "path_off decreases at leaf 1" in msg
    for field, value in (("from", 64), ("to", 64), ("from", 255), ("promo", 1), ("promo", 6)):
        f2 = flat.copy()
        f2[field][4] = value
        rc, msg, _ = _raw_predict_path(e, [0, 1, 2], f2, off)
        assert rc == SC_E_INVAL and "path[4]" in msg, (field, value, msg)
        # and in a root: sc_set_roots rejects it before any launch and keeps the table
        rf, ro = _flat(roots)
        rf[field][7] = value
        rc = L.sc_set_roots(e.handle, 3, rf.ctypes.data, ro.ctypes.data)
        assert rc == SC_E_INVAL and "stack[7]" in L.sc_last_error().decode()
        assert _raw_predict_path(e, [0, 1, 2], flat, off)[0] == 0
    # n_hist counts the whole game: root 0 has 5 plies, so its leaves take up to min(8, 5 + path + 1)
    for nh, ok in (([8, 8, 8], True), ([7, 3, 1], True), ([0, 1, 1], False), ([9, 1, 1], False)):
        rc, msg, _ = _raw_predict_path(e, [0, 1, 2], flat, off, n_hist=nh)
        assert (rc == 0) == ok and (ok or "n_hist[0]" in msg), (nh, msg)
    e.set_roots([g[:2]])
    rc, msg, _ = _raw_predict_path(e, [0], *_flat([g[2:4]]), n_hist=[6])
    assert rc == SC_E_INVAL and "n_hist[0] = 6 is not in 1..5" in msg
    # root plus path longer than SC_MAX_STACK: a 1000-ply root takes at most 24 more plies
    long = KNIGHTS * 250
    e.set_roots([long, []])
    assert _raw_predict_path(e, [0], *_flat([KNIGHTS * 6]))[0] == 0
    rc, msg, _ = _raw_predict_path(e, [1, 0], *_flat([[], KNIGHTS * 6 + KNIGHTS[:1]]))
    assert rc == SC_E_INVAL and "leaf 1 has 1025 plies, more than SC_MAX_STACK" in msg, msg
    rc, msg = _raw_set_roots(e, [[], KNIGHTS * 256 + KNIGHTS[:1]])
    assert rc == SC_E_INVAL and "root 1 has 1025 plies, more than SC_MAX_STACK" in msg, msg
    # n > max_batch, NULL arguments, n_roots > max_batch
    rc = e.predict_path([0] * 9, [[]] * 9, check=False)[0]
    assert rc == SC_E_INVAL
    z = np.zeros(4, np.float32)
    assert L.sc_predict_path(e.handle, 1, None, None, off.ctypes.data, None, None, z.ctypes.data, z.ctypes.data,
                             z.ctypes.data, z.ctypes.data, None) == SC_E_INVAL
    assert _raw_set_roots(e, [[]] * 9)[0] == SC_E_INVAL
    assert L.sc_set_roots(e.handle, 1, None, None) == SC_E_INVAL
    e.close()


def test_path_rejections(engine, random_games):
    """a move rejected in the path: the message names the leaf and the ply from the game start, and the outputs are
    written as sc_predict_stack writes them for root ++ path"""
    import scb200

    L = scb200.load_library()
    for stack, ply, words in _rejections():
        for cut in range(0, ply + 1):  # the rejected move is in the path, at every distance from the root
            roots = [[], stack[:cut], _uci("d2d4")]
            engine.set_roots(roots)
            paths = [[], stack[cut:], []]
            rc, msg, got = _raw_predict_path(engine, [0, 1, 2], *_flat(paths))
            assert rc == SC_E_INVAL and f"sc_predict_path: leaf 1, ply {ply}" in msg and words in msg, (cut, msg)
            exp = engine.predict_stack([r + p for r, p in zip(roots, paths)], positions=True, check=False)
            assert exp[0] == SC_E_INVAL
            assert L.sc_last_error().decode().replace("sc_predict_stack", "sc_predict_path") == msg
            _assert_same(got, exp[1:], (stack, cut))


def test_roots_persist(blob, random_games):
    """a second sc_set_roots replaces the table; roots survive sc_predict, sc_predict_stack and sc_eval calls in between
    (including calls that grow the replay scratch); two engines keep separate tables"""
    import scb200

    rng = np.random.RandomState(21)
    e1 = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 2048)
    e2 = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 2048)
    roots_a, leaf_a, paths_a = _leaf_batch(random_games, 200, 50, rng)
    roots_b, leaf_b, paths_b = _leaf_batch(random_games[::-1], 200, 70, rng)
    _check_against_stack(e1, roots_a, leaf_a, paths_a, what="a")
    _check_against_stack(e2, roots_b, leaf_b, paths_b, what="b")
    ref_a = [np.copy(x) for x in e1.predict_path(leaf_a, paths_a, positions=True)]
    # other calls on e1, with bigger batches and longer games than the path calls use
    stacks = [g for g in random_games] * 40
    e1.predict_stack(stacks[:2048])
    long = [g[:100] for g in random_games if len(g) > 100][:16]
    pos = np.array([scb200.rules_probe(g)[1] for g in long], dtype=scb200.POSITION_DTYPE)
    e1.predict(pos)
    mv = [scb200.rules_probe(g)[0] for g in long]
    off = np.zeros(17, dtype=np.int32)
    off[1:] = np.cumsum([len(m) for m in mv])
    moves = np.zeros(int(off[-1]), dtype=scb200.MOVE_DTYPE)
    for m, o in zip(mv, off[:-1]):
        for k, x in enumerate(m):
            moves[o + k] = (x[0], x[1], x[2], 0)
    e1.eval(pos, moves, off)
    _check_against_stack(e2, roots_b, leaf_b, paths_b, what="b after a's calls", set_roots=False)
    _assert_same(e1.predict_path(leaf_a, paths_a, positions=True), ref_a, "a after other calls")
    # e2's table replaced by a smaller one: old indices past it are rejected, the new ones read the new games
    e2.set_roots(roots_a[:10])
    assert e2.predict_path([10], [[]], check=False)[0] == SC_E_INVAL
    sel = [i for i in range(len(leaf_a)) if leaf_a[i] < 10]
    _check_against_stack(e2, roots_a[:10], [leaf_a[i] for i in sel], [paths_a[i] for i in sel], what="replaced",
                         set_roots=False)
    _check_against_stack(e1, roots_a, leaf_a, paths_a, what="a again", set_roots=False)
    e1.close()
    e2.close()


def test_garbage_paths_stay_in_their_slots(engine, random_games):
    """random-byte paths next to real leaves: the real leaves are intact and nothing is written past row n"""
    rng = np.random.RandomState(23)
    roots, leaf_root, real = _leaf_batch(random_games, 1024, 64, rng)
    paths = []
    for i in range(1024):
        if i % 2 == 0:
            paths.append(real[i])
        else:
            ln = rng.randint(0, 31)
            paths.append(list(zip(rng.randint(0, 64, ln), rng.randint(0, 64, ln), rng.choice([0, 2, 3, 4, 5], ln))))
    engine.set_roots(roots)
    for n in (1024, 40):  # device buffers, and the pinned staging buffer
        rc, msg, got = _raw_predict_path(engine, leaf_root[:n], *_flat(paths[:n]), guard_rows=3)
        assert rc in (0, SC_E_INVAL), msg
        cnt = got[1]
        assert ((cnt >= 0) & (cnt <= 256)).all()
        even = list(range(0, n, 2))
        exp = engine.predict_stack([roots[leaf_root[i]] + real[i] for i in even], positions=True)
        _assert_same(tuple(a[even] for a in got), exp, ("garbage", n))
    # the engine answers a normal call afterwards
    _check_against_stack(engine, roots, leaf_root[:64:2], real[:64:2], what="after garbage", set_roots=False)


def test_shim_root_policy(engine, sample_games, capsys):
    """INTEGRATION.md's policy for the Rust shim, emulated over every ply of a few sample games with two leaves per
    ply at random depths 0..12: reuse the cached root while it is a prefix of the leaf's stack and at most 48 plies
    behind, else store the stack minus its last 16 plies.  One-leaf calls, bit-identical to sc_predict_stack, and
    about one sc_set_roots per 30 plies"""
    import scb200

    rng = np.random.RandomState(31)
    games = [_uci(g["uci"]) for g in sample_games["games"]]
    games = sorted(games, key=len)[-4:]
    cached, n_set, n_calls, plies = None, 0, 0, 0
    for g in games:
        plies += len(g)
        for t in range(len(g) + 1):
            for _ in range(2):
                stack = list(g[:t])
                for _ in range(rng.randint(0, 13)):
                    mv = scb200.rules_probe(stack)[0]
                    if len(mv) == 0:
                        break
                    stack.append(tuple(int(x) for x in mv[rng.randint(len(mv))]))
                if cached is None or stack[: len(cached)] != cached or len(stack) - len(cached) > 48:
                    cached = stack[: max(0, len(stack) - 16)]
                    engine.set_roots([cached])
                    n_set += 1
                got = engine.predict_path([0], [stack[len(cached) :]], positions=True)
                exp = engine.predict_stack([stack], positions=True)
                _assert_same(got, exp, (t, len(stack)))
                n_calls += 1
    with capsys.disabled():
        print(f"\nshim policy: {n_calls} predict calls over {plies} plies of {len(games)} games, {n_set} sc_set_roots "
              f"(one per {plies / n_set:.1f} plies)")
    assert n_set <= plies / 20 + len(games)
