"""CPU tests of the chess oracle against everything the reference pins (SURVEY 4, 8c)."""
import hashlib
import os

import numpy as np
import pytest

START_ORDER = "g1h3 g1f3 b1c3 b1a3 h2h3 g2g3 f2f3 e2e3 d2d3 c2c3 b2b3 a2a3 h2h4 g2g4 f2f4 e2e4 d2d4 c2c4 b2b4 a2a4".split()
BLACK_ORDER = "g8h6 g8f6 b8c6 b8a6 h7h6 g7g6 f7f6 e7e6 d7d6 c7c6 b7b6 a7a6 h7h5 g7g5 f7f5 e7e5 d7d5 c7c5 b7b5 a7a5".split()
START_INDEX = [494, 501, 129, 136, 1095, 1022, 949, 876, 803, 730, 657, 584, 1096, 1023, 950, 877, 804, 731, 658, 585]


def test_move_order_notebook_goldens(co):
    # notebooks/verify_model.ipynb:142-161 and :454-473
    g = co.Game()
    assert g.legal_uci() == START_ORDER
    g.push("g2g3")
    assert g.legal_uci() == BLACK_ORDER


def test_move_index_known_answers(co):
    # SURVEY appendix A.1 (derived from queenmoves.rs / knightmoves.rs / underpromotions.rs)
    g = co.Game()
    assert [int(i) for i in g.move_indices()] == START_INDEX
    g.push("g2g3")
    assert [int(i) for i in g.move_indices()] == START_INDEX  # rank flip for Black
    W, B = 1, 0
    mi = lambda u, t: co.move_index(co.parse_uci(u), t)
    assert mi("e1g1", W) == 307 and mi("e1c1", W) == 335 and mi("e8g8", B) == 307
    assert mi("a7a8q", W) == 3504 and mi("a7b8n", W) == 3574 and mi("h2g1r", B) == 4081
    # notebooks/visualize_mcts.ipynb:992-1001: 751 <-> (rank 1, file 2, type 21)
    assert 1 * 584 + 2 * 73 + 21 == 751
    assert mi("c2c5", W) != 751 and mi("c2f2", W) == 1 * 584 + 2 * 73 + 2 * 7 + 2
    # type 21 = direction 3 (d_rank -1, d_file +1), distance 1: c2 -> d1
    assert mi("c2d1", W) == 751


def test_move_index_exhaustive_range_and_injective(co):
    # every geometrically valid (from, to, promo) maps into [0, 4672) and distinct moves from the
    # same square get distinct indices
    for turn in (0, 1):
        for f in range(64):
            seen = {}
            for t in range(64):
                if t == f:
                    continue
                dr, df = (t >> 3) - (f >> 3), (t & 7) - (f & 7)
                queen = dr == 0 or df == 0 or abs(dr) == abs(df)
                knight = sorted((abs(dr), abs(df))) == [1, 2]
                promos = [0]
                fr = (f >> 3) if turn else 7 - (f >> 3)
                tr = (t >> 3) if turn else 7 - (t >> 3)
                if fr == 6 and tr == 7 and abs(df) <= 1:
                    promos = [0, 2, 3, 4, 5]
                for p in promos:
                    idx = co.move_index((f, t, p), turn)
                    if not (queen or knight):
                        assert idx == -1
                        continue
                    if knight and p:
                        continue
                    assert 0 <= idx < 4672
                    key = (t, p if p in (2, 3, 4) else 0)
                    assert seen.setdefault(idx, key) == key


def test_root_planes_known_answer(co):
    # SURVEY appendix A.2
    g = co.Game()
    planes, meta = g.encode()
    assert planes.shape == (8, 8, 112) and planes.dtype == np.int8
    assert list(meta) == [1, 1, 1, 1, 1, 1, 0]
    assert planes[:, :, 14:].sum() == 0
    assert (planes[1, :, 0] == 1).all() and planes[:, :, 0].sum() == 8
    assert planes[0, 1, 1] == 1 and planes[0, 6, 1] == 1 and planes[:, :, 1].sum() == 2
    assert planes[0, 4, 5] == 1 and planes[7, 4, 11] == 1 and planes[0, 3, 4] == 1
    assert planes[:, :, 12].sum() == 0 and planes[:, :, 13].sum() == 0
    g.push("g2g3")
    planes, meta = g.encode()
    assert list(meta) == [0, 1, 1, 1, 1, 1, 0]
    assert (planes[1, :, 0] == 1).all()          # Black's pawns shown on rank index 1
    assert planes[0, 4, 5] == 1                  # Black king at (0, 4) after the flip
    assert planes[5, 6, 6] == 1 and planes[6, 6, 6] == 0 and planes[:, :, 6].sum() == 8
    assert (planes[6, :, 14 + 6] == 1).all()     # slot 1 = start position, also flipped
    assert planes[:, :, 28:].sum() == 0
    # history stops at the tree root
    p0, _ = g.encode(node_depth=0)
    assert p0[:, :, 14:].sum() == 0 and (p0[:, :, :14] == planes[:, :, :14]).all()


def test_meta_examples(co, sample_games):
    # notebooks/verify_model.ipynb:34 style: [turn, fullmove, castling x4, halfmove]
    g = co.Game()
    for u in sample_games["games"][1]["uci"].split()[:50]:
        g.push(u)
    _, meta = g.encode()
    assert meta[0] == 1 and meta[1] == 26


def test_perft(co):
    assert [co.Game().perft(d) for d in range(1, 5)] == [20, 400, 8902, 197281]
    cases = [
        ("r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1", [48, 2039, 97862]),
        ("8/2p5/3p4/KP5r/1R3p1k/8/4P1P1/8 w - - 0 1", [14, 191, 2812, 43238]),
        ("r3k2r/Pppp1ppp/1b3nbN/nP6/BBP1P3/q4N2/Pp1P2PP/R2Q1RK1 w kq - 0 1", [6, 264, 9467]),
        ("rnbq1k1r/pp1Pbppp/2p5/8/2B5/8/PPP1NnPP/RNBQK2R w KQ - 1 8", [44, 1486, 62379]),
        ("r4rk1/1pp1qppp/p1np1n2/2b1p1B1/2B1P1b1/P1NP1N2/1PP1QPPP/R4RK1 w - - 0 10", [46, 2079, 89890]),
    ]
    for fen, exp in cases:
        g = co.Game(fen)
        assert [g.perft(d + 1) for d in range(len(exp))] == exp


def test_chess_fast_fen_move_count(co):
    # the only FEN in the reference's own #[test] (src/chess_fast.rs:84-98)
    g = co.Game("1k1r4/1r5p/p4n1P/1ppP1P2/PP6/4PP1b/3B4/R1N1K3 b - - 0 39")
    mv = g.legal_uci()
    assert len(mv) == len(set(mv)) and len(mv) > 20 and "b5a4" in mv and "h3f1" in mv


def test_max_moves_position(co):
    g = co.Game("R6R/3Q4/1Q4Q1/4Q3/2Q4Q/Q4Q2/pp1Q4/kBNN1KB1 w - - 0 1")
    assert len(g.legal_moves()) == 218


def test_sample_games_replay_digest(co, sample_games):
    # replay of the 60 games shipped in py/validation/sample.csv (stored as UCI): every move must be
    # oracle-legal, and planes/meta/indices must hash to the committed digest
    assert sample_games["totals"]["plies"] == 3539 and sample_games["totals"]["mate"] == 11
    for game in sample_games["games"]:
        g = co.Game()
        h = hashlib.sha256()
        for u in game["uci"].split():
            planes, meta = g.encode()
            idx = g.move_indices()
            assert (idx >= 0).all() and len(set(idx.tolist())) == len(idx)
            h.update(planes.tobytes()); h.update(meta.tobytes()); h.update(idx.tobytes())
            assert u in g.legal_uci()
            g.push(u)
        assert h.hexdigest() == game["sha256"]


def test_sample_csv_san_resolution(co, sample_games):
    """The oracle's SAN parser on the 60 games of the reference's py/validation/sample.csv: tests/golden/sample_san.json
    holds either the CSV's own text (oracle/make_golden_chess.py) or, as its `source` says, a reconstruction written
    without the oracle (oracle/make_golden_san.py).  The totals are the ones recorded from the CSV."""
    import json

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sample_san.json")) as f:
        rows = json.load(f)["games"]
    assert len(rows) == 60
    sans = [s for row in rows for s in row["moves"].split()]
    tot = sample_games["totals"]
    assert len(sans) == tot["plies"] and sum(s[-1] in "+#" for s in sans) == tot["check"]
    assert sum(s.endswith("#") for s in sans) == tot["mate"]
    assert sum(s.startswith("O-O") for s in sans) == tot["castle"] and sum("=" in s for s in sans) == tot["promo"]
    ep = 0
    for row, game in zip(rows, sample_games["games"]):
        assert row["id"] == game["id"]
        g = co.Game()
        ucis = []
        for san in row["moves"].split():
            m = g.parse_san(san)
            f, t = int(m[0]), int(m[1])
            ep += abs(g.piece_at(f)) == 1 and (f & 7) != (t & 7) and g.piece_at(t) == 0
            g.push(m)
            ucis.append(co.uci(m))
            assert g.is_check() == (san[-1] in "+#")
            assert (len(g.legal_moves()) == 0 and g.is_check()) == san.endswith("#")
        assert " ".join(ucis) == game["uci"]
    assert ep == tot["ep"]


def test_repetition_flags(co):
    g = co.Game()
    for u in "g1f3 g8f6 f3g1 f6g8".split():
        g.push(u)
    assert g.is_repetition(2) and not g.is_repetition(3)
    planes, _ = g.encode()
    assert (planes[:, :, 12] == 1).all() and (planes[:, :, 13] == 0).all()
    assert (planes[:, :, 14 + 12] == 0).all()          # previous slot had not repeated yet
    for u in "g1f3 g8f6 f3g1 f6g8".split():
        g.push(u)
    assert g.is_repetition(3)
    planes, _ = g.encode()
    assert (planes[:, :, 13] == 1).all()
    assert g.outcome(claim_draw=True) == (7, -1)       # Termination::ThreefoldRepetition
    # a pawn move is irreversible: no repetition across it
    g2 = co.Game()
    for u in "g1f3 g8f6 e2e3 f6g8 f3g1".split():
        g2.push(u)
    assert not g2.is_repetition(2)


def test_castling_rights_and_en_passant(co):
    g = co.Game()
    for u in "e2e4 e7e5 g1f3 b8c6 f1c4 f8c5 e1g1".split():
        g.push(u)
    _, meta = g.encode()
    assert list(meta[:6]) == [0, 4, 1, 1, 0, 0]       # Black to move keeps both, White lost both
    assert g.piece_at(co.sq_parse("g1")) == 6 and g.piece_at(co.sq_parse("f1")) == 4
    g = co.Game()
    for u in "e2e4 a7a6 e4e5 d7d5".split():
        g.push(u)
    assert "e5d6" in g.legal_uci()
    g.push("e5d6")
    assert g.piece_at(co.sq_parse("d5")) == 0 and g.piece_at(co.sq_parse("d6")) == 1


def test_outcomes(co):
    g = co.Game()
    for u in "f2f3 e7e5 g2g4 d8h4".split():
        g.push(u)
    assert g.outcome() == (1, 0) and len(g.legal_moves()) == 0   # checkmate, Black wins
    assert co.Game("7k/5Q2/6K1/8/8/8/8/8 b - - 0 1").outcome() == (2, -1)   # stalemate
    assert co.Game("8/8/4k3/8/8/3K4/8/8 w - - 0 1").outcome() == (3, -1)     # insufficient material
    assert co.Game("8/8/4k3/8/8/3K4/7R/8 w - - 100 80").outcome() == (6, -1)  # fifty moves (claim)
    assert co.Game().outcome() is None


def test_post_process_matches_numpy_restatement(co):
    import net

    rng = np.random.RandomState(0)
    logp = np.log(rng.dirichlet(np.ones(4672))).astype(np.float32)
    idx = rng.choice(4672, size=31, replace=False).astype(np.int32)
    a = co.post_process(logp, idx)
    b = net.priors_from_logp(logp, idx)
    assert np.allclose(a, b, rtol=0, atol=1e-7)
    assert abs(a.sum() - a.sum() / (a.sum() + 0)) < 1 and a.sum() < 1.0


def test_sequential_search_invariants(co):
    # SURVEY appendix A.4: after R rollouts root N = R and sum of child N = R - 1
    t = co.Tree()
    t.search(40, 2.5)
    mv, n_act, q, u = t.root_children()
    assert t.root_n() == 40 and n_act.sum() == 39 and len(mv) == 20
    assert t.n_evals <= t.n_predicts
    before = n_act.copy()
    i = t.step_argmax()
    assert i == int(np.argmax(before)) and t.root_n() == 0 and t.game.ply == 1
    # determinism
    t2 = co.Tree()
    t2.search(40, 2.5)
    assert (t2.root_children()[1] == before).all()


def test_encode_steps_literal_restatement(co):
    """`chess_encode_steps` restated literally (double rotation under apply_mirror): its planes equal
    `_encode`'s with and without the mirror; only the meta differs (rotated board's meta)."""
    g = co.Game()
    steps = []
    rng = np.random.RandomState(3)
    for _ in range(30):
        mv = g.legal_moves()
        m = mv[rng.randint(len(mv))]
        steps.append((tuple(int(x) for x in m), [(tuple(int(x) for x in c), int(rng.randint(0, 9))) for c in mv]))
        g.push(m)
    plain = co.encode_steps(steps, False)
    mirr = co.encode_steps(steps, True)
    g = co.Game()
    for (mv, _), (p0, m0, d0, i0), (p1, m1, d1, i1) in zip(steps, plain, mirr):
        planes, meta = g.encode()
        assert np.array_equal(p0, planes) and np.array_equal(m0, meta)
        assert np.array_equal(p1, planes) and i0 == i1 and np.array_equal(d0, d1)
        assert m1[0] == 1 - meta[0] and m1[1] == meta[1] + (1 if meta[0] == 1 else 0)
        assert list(m1[2:6]) == [meta[4], meta[5], meta[2], meta[3]] and m1[6] == meta[6]
        assert i0 == [int(x) for x in g.move_indices()]
        assert abs(d0.sum() - 1.0) < 1e-4 or d0.sum() == 0
        g.push(mv)


PYCHESS_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pychess_golden.json.gz")


def _check_games(co, games, check_oracle: bool):
    """Holds the product's native rules (and, with check_oracle, the C oracle) to per-ply records in the format of
    oracle/make_golden_pychess.py."""
    import scb200

    n = 0
    for game in games:
        fen = game["fen"]
        g = co.Game(fen) if fen else co.Game()
        hist = []
        for ply, rec in enumerate(game["plies"]):
            where = (game["source"], fen, ply)
            if check_oracle:
                assert g.legal_uci() == rec["legal"], where
                assert g.is_repetition(2) == rec["rep2"] and g.is_repetition(3) == rec["rep3"], where
                assert [int(v) for v in g.encode()[1]] == rec["meta"], where
                oc = g.outcome(True)
                assert (None if oc is None else [int(oc[0]), int(oc[1])]) == rec["outcome"], where
            mv, pos, (term, win) = scb200.rules_probe(hist, fen)
            assert [co.uci(m) for m in mv] == rec["legal"], where
            assert [int(v) for v in pos["meta"]] == rec["meta"], where
            assert bool(int(pos["slot"][0][7]) & 1) == rec["rep2"] and bool(int(pos["slot"][0][7]) & 2) == rec["rep3"], where
            assert (None if term == 0 else [term, win]) == rec["outcome"], where
            n += 1
            if ply < len(game["moves"]):
                g.push(game["moves"][ply])
                hist.append(tuple(int(v) for v in co.parse_uci(game["moves"][ply])))
    return n


def _edge_fens():
    import re

    src = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle", "make_golden_pychess.py")).read()
    block = src[src.index("EDGE_FENS = ["):src.index("]", src.index("EDGE_FENS = ["))]
    return re.findall(r'"([^"]+ [wb] [KQkq-]+ [a-h1-8-]+ \d+ \d+)"', block)


def test_native_rules_equal_oracle_on_the_golden_generators_cases(co):
    """The same games the python-chess generator plays (edge-case FENs, repetition shuffle, a long rook ending), recorded
    with the C ORACLE instead, in the generator's format: the product's independent rules engine must agree ply by ply
    on move order, repetition flags, meta and outcome(claim_draw=True).  (Differential test; the python-chess pin itself
    is test_rules_against_python_chess_goldens.)"""
    fens = _edge_fens()
    assert len(fens) >= 20
    rng = np.random.RandomState(12)

    def rec(g):
        oc = g.outcome(True)
        return {"legal": g.legal_uci(), "rep2": g.is_repetition(2), "rep3": g.is_repetition(3),
                "meta": [int(v) for v in g.encode()[1]], "outcome": None if oc is None else [int(oc[0]), int(oc[1])]}

    def play(fen, n_plies, moves=None):
        g = co.Game(fen) if fen else co.Game()
        plies, ucis = [rec(g)], []
        for k in range(n_plies):
            legal = g.legal_uci()
            if not legal:
                break
            u = moves[k] if moves else legal[rng.randint(len(legal))]
            ucis.append(u)
            g.push(u)
            plies.append(rec(g))
        return {"fen": fen, "moves": ucis, "plies": plies, "source": "oracle"}

    games = [play(f, 50) for f in fens for _ in range(2)]
    games.append(play(None, 20, ["g1f3", "g8f6", "f3g1", "f6g8"] * 5))
    games.append(play("8/8/8/4k3/8/8/3RK3/8 w - - 0 1", 320))
    n = _check_games(co, games, check_oracle=False)
    assert n > 2000
    outcomes = {tuple(p["outcome"]) for g in games for p in g["plies"] if p["outcome"]}
    assert {1, 2, 3, 5, 6, 7} <= {o[0] for o in outcomes} | {4}      # every termination kind but (maybe) 75-move is met
    assert any(p["rep3"] for g in games for p in g["plies"])


def test_rules_against_python_chess_goldens(co):
    """Rows a6 / c of SURVEY section 8: everything the hot path takes from python-chess (legal-move ORDER,
    is_repetition(2/3), castling-rights view, clocks, outcome(claim_draw=True)) for both rule engines -- the C oracle and
    the product's native rules -- against a dump made by python-chess itself (oracle/make_golden_pychess.py).
    python-chess cannot be installed in the offline build container; until somebody with python-chess runs the generator
    and commits its output this test reports the rules as UNPINNED (an expected failure, not a pass)."""
    import gzip
    import json

    if not os.path.exists(PYCHESS_GOLDEN):
        pytest.xfail("PARITY UNPINNED: tests/golden/pychess_golden.json.gz is absent -- run oracle/make_golden_pychess.py "
                     "where python-chess 1.11.1 is installed; until then move order, repetition flags and draw claims of "
                     "both rule engines are checked only against each other, perft tables and the reference's two "
                     "notebook move lists")
    with gzip.open(PYCHESS_GOLDEN, "rt") as f:
        gold = json.load(f)
    assert gold["n_plies"] >= 13000
    assert _check_games(co, gold["games"], check_oracle=True) == gold["n_plies"]


def test_move_order_of_the_reference_notebook_trace(co):
    """notebooks/verify_model.ipynb holds the first ten plies of a trace the reference produced on real python-chess:
    per ply the root's children in `predict`'s order = python-chess' legal-move generation order.  Both rule engines must
    reproduce all ten lists (19 - 36 moves; queen sorties, pawn captures) while replaying the moves, and the 40-ply game of
    notebooks/visualize_mcts.ipynb must replay as legal moves (tests/golden/notebook_traces.json, made by
    oracle/make_golden_notebooks.py).  These are the only python-chess-made move lists available offline."""
    import json

    import scb200

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "notebook_traces.json")) as f:
        gold = json.load(f)
    g = co.Game()
    hist = []
    assert len(gold["verify_model_trace"]) == 10
    for ply, st in enumerate(gold["verify_model_trace"]):
        assert g.legal_uci() == st["children"], ply
        mv, pos, _ = scb200.rules_probe(hist)
        assert [co.uci(m) for m in mv] == st["children"], ply
        assert st["move"] in st["children"]
        g.push(st["move"])
        hist.append(tuple(int(v) for v in co.parse_uci(st["move"])))
    g = co.Game()
    hist = []
    for u in gold["visualize_mcts_game"]:
        assert u in g.legal_uci(), u
        mv, _, _ = scb200.rules_probe(hist)
        assert u in [co.uci(m) for m in mv]
        g.push(u)
        hist.append(tuple(int(v) for v in co.parse_uci(u)))
