"""sc_evaluator_*: many threads, each submitting one leaf at a time, share one engine through a batching evaluator with
a root slot per game.

A leaf's result must not depend on the pass it lands in, so every output is compared bit for bit with sc_predict_stack
on root ++ path (itself checked against sc_predict_path and the host rules in test_gpu_predict_path.py /
test_gpu_predict_stack.py), computed on the same engine before the evaluator takes it over.
"""
import json
import os
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = ("SC_MODE_FP32", "SC_MODE_BF16", "SC_MODE_FP32_FFMA", "SC_MODE_FP16")
SC_E_INVAL, SC_E_STATE = -1, -5


@pytest.fixture(scope="module")
def blob(tmp_path_factory):
    import net
    import scb200

    p = str(tmp_path_factory.mktemp("w") / "n2.scw")
    scb200.write_blob(net.perturb_norm_params(net.init_state_dict(2, 7), 1234), p)
    return p


def _random_games(n_games, max_plies, seed):
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


def _sq(s):
    return (int(s[1]) - 1) * 8 + ord(s[0]) - ord("a")


def _uci(text):
    return [(_sq(u[:2]), _sq(u[2:4]), " pnbrqk".index(u[4]) if len(u) > 4 else 0) for u in text.split()]


@pytest.fixture(scope="module")
def leaves(sample_games):
    """(roots, [(slot, path)]): 8 random-play roots and 8 sample-game prefixes, 8 leaves of 0..30 plies on each"""
    import scb200

    roots = _random_games(8, 90, seed=3)
    sample = [_uci(g["uci"]) for g in sample_games["games"]]
    roots += [sample[k % len(sample)][: (0, 1, 9, 20, 33, 47, 60, 400)[k]] for k in range(8)]
    rng = np.random.RandomState(11)
    out = []
    for g, root in enumerate(roots):
        for k in range(8):
            hist, path = list(root), []
            want = (0, 1, 2, 5, 12, 20, 30, int(rng.randint(31)))[k]
            while len(path) < want:
                mv = scb200.rules_probe(hist)[0]
                if len(mv) == 0:
                    break
                m = tuple(int(x) for x in mv[rng.randint(len(mv))])
                hist.append(m)
                path.append(m)
            out.append((g, path))
    return roots, out


def _reference(eng, roots, specs):
    """predict_stack on root ++ path, one leaf at a time (check=False: rc first)"""
    return [eng.predict_stack([list(roots[g]) + list(p)], positions=True, check=False) for g, p in specs]


def _same(got, ref):
    """evaluator predict(positions=True, check=False) against one leaf of predict_stack(check=False), bit for bit"""
    rc, moves, cnt, priors, value, pos = got
    rrc, rmoves, rcnt, rpriors, rvals, rpos = ref
    assert rc == rrc
    assert cnt == rcnt[0]
    assert np.array_equal(moves[:cnt], rmoves[0][:cnt])
    assert np.array_equal(priors[:cnt].view(np.uint32), rpriors[0][:cnt].view(np.uint32))
    assert np.float32(value).view(np.uint32) == rvals[0:1].view(np.uint32)[0]
    assert pos.tobytes() == rpos[0].tobytes()


def _run_threads(n, fn):
    errs = []

    def wrap(t):
        try:
            fn(t)
        except BaseException as ex:  # noqa: BLE001 - reported below
            errs.append(ex)

    th = [threading.Thread(target=wrap, args=(t,)) for t in range(n)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]


@pytest.mark.parametrize("mode", MODES)
def test_leaves_bit_identical_to_predict_stack(blob, leaves, mode):
    import scb200

    roots, specs = leaves
    eng = scb200.Engine(blob, 0, getattr(scb200, mode), 512)
    ref = _reference(eng, roots, specs)
    ev = scb200.Evaluator(eng, len(roots))
    for g, r in enumerate(roots):
        ev.set_root(g, r)
    for n_threads in (1, 8, 64, 512):
        got = [None] * max(len(specs), n_threads)

        def work(t):
            for i in range(t, max(len(specs), n_threads), n_threads):
                g, p = specs[i % len(specs)]
                got[i] = ev.predict(g, p, positions=True, check=False)

        _run_threads(n_threads, work)
        for i, r in enumerate(got):
            _same(r, ref[i % len(specs)])
    st = ev.stats()
    print(mode, st)
    assert st["largest_batch"] > 1 and st["leaves"] == len(specs) * 3 + 512
    ev.close()
    eng.close()


def test_root_slots(blob, leaves):
    import scb200

    roots, specs = leaves
    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 64)
    ref = _reference(eng, roots, specs)
    ev = scb200.Evaluator(eng, 2 * len(roots))
    # slot g: the whole game; slot g + 16: the same game in steps of 0..7 plies
    for g, r in enumerate(roots):
        ev.set_root(g, r)
        ev.set_root(g + len(roots), [])
        k, j = 0, g
        while k < len(r):
            step = j % 8  # 0 once in every 8 steps: an empty extension
            j += 1
            ev.extend_root(g + len(roots), r[k : k + step])
            k += step
    for i, (g, p) in enumerate(specs):
        _same(ev.predict(g, p, positions=True, check=False), ref[i])
        _same(ev.predict(g + len(roots), p, positions=True, check=False), ref[i])

    # re-rooting slot 0 again and again while other threads' leaves on the other slots are in flight
    stop = threading.Event()

    def reroot():
        while not stop.is_set():
            ev.set_root(0, roots[1])
            ev.set_root(0, roots[0])

    th = threading.Thread(target=reroot)
    th.start()
    try:
        others = [(i, s) for i, s in enumerate(specs) if s[0] != 0]

        def work(t):
            for i, (g, p) in others[t::16]:
                _same(ev.predict(g, p, positions=True, check=False), ref[i])

        _run_threads(16, work)
    finally:
        stop.set()
        th.join()

    # documented errors
    long_root = (list(roots[0]) + [(6, 21, 0), (21, 6, 0), (62, 45, 0), (45, 62, 0)] * 300)[: scb200.SC_MAX_STACK + 1]
    assert ev.set_root(3, long_root, check=False) == SC_E_INVAL
    assert "slot 3 has 1025 plies, more than SC_MAX_STACK = 1024" in scb200.last_error()
    _same(ev.predict(3, specs[24][1], positions=True, check=False), ref[24])  # slot 3 left as it was
    assert ev.set_root(2 * len(roots), [], check=False) == SC_E_INVAL and "slot" in scb200.last_error()
    assert ev.predict(-1, [], check=False)[0] == SC_E_INVAL
    # e2e4 e7e5 then a white move from an empty square at ply 2
    assert ev.set_root(4, [(12, 28, 0), (52, 36, 0), (20, 28, 0)], check=False) == SC_E_INVAL
    assert "sc_evaluator_set_root: slot 4, ply 2: move rejected" in scb200.last_error()
    assert ev.predict(4, [], check=False)[0] == SC_E_STATE and "slot 4 has no root" in scb200.last_error()
    assert ev.extend_root(4, [(12, 28, 0)], check=False) == SC_E_STATE
    ev.set_root(5, [])
    assert ev.extend_root(5, [(12, 28, 0), (12, 20, 0)], check=False) == SC_E_INVAL
    assert "slot 5, ply 1: move rejected" in scb200.last_error()
    assert ev.predict(5, [], check=False)[0] == SC_E_STATE
    ev.close()
    eng.close()


def test_error_isolation(blob, leaves):
    """one pass mixing rejected paths, random-byte paths and real leaves: only the bad callers fail"""
    import scb200

    roots, specs = leaves
    rng = np.random.RandomState(5)
    mixed = list(specs)
    for k in range(24):
        g = int(rng.randint(len(roots)))
        rand = [(int(rng.randint(64)), int(rng.randint(64)), int(rng.choice([0, 0, 0, 2, 3, 4, 5])))
                for _ in range(1 + rng.randint(12))]
        mixed.append((g, rand if k % 2 else [(12, 28, 0)] * 3))
    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 256)
    ref = _reference(eng, roots, mixed)
    ev = scb200.Evaluator(eng, len(roots))
    for g, r in enumerate(roots):
        ev.set_root(g, r)
    got, msg = [None] * len(mixed), [None] * len(mixed)

    def work(t):
        for i in range(t, len(mixed), 64):
            got[i] = ev.predict(mixed[i][0], mixed[i][1], positions=True, check=False)
            msg[i] = scb200.last_error() if got[i][0] else None

    _run_threads(64, work)
    n_bad = 0
    for i, (g, p) in enumerate(mixed):
        _same(got[i], ref[i])
        if got[i][0]:
            n_bad += 1
            assert msg[i].startswith(f"sc_evaluator_predict: slot {g}, ply ")
            assert "move rejected" in msg[i] or "pseudo-legal" in msg[i]
    assert n_bad >= 12 and ev.stats()["largest_batch"] > 1
    ev.close()
    eng.close()


def test_reference_search_through_the_evaluator(tmp_path, blob):
    """16 games of mcts::mcts / mcts::step on 16 threads through one evaluator: in fp32 with the seed-0 19-block net
    and the configs[0] settings each replays the golden game; in bf16 each equals sc_game_selfplay's game alone"""
    import scb200

    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "search_cfg1.json")))
    cfg = gold["config"]
    blob19 = str(tmp_path / "seed0.scw")
    scb200.write_blob(scb200.random_init_state_dict(cfg["n_res_blocks"], 0), blob19)
    eng = scb200.Engine(blob19, 0, scb200.SC_MODE_FP32, 16)
    traces, counts = scb200.game_selfplay_many(eng, [0] * 16, rollout_num=cfg["rollout_num"],
                                               num_steps=cfg["num_steps"], cpuct=cfg["cpuct"])
    print("fp32, 16 games:", counts)
    assert counts["largest_batch"] > 1
    for tr in traces:
        assert len(tr["steps"]) == len(gold["steps"])
        for (mv, q, ch), ref in zip(tr["steps"], gold["steps"]):
            assert mv == ref["move"]
            assert [(c[0], c[1]) for c in ch] == [(c[0], c[1]) for c in ref["children"]]
            assert max(abs(c[2] - r[2]) for c, r in zip(ch, ref["children"])) < 1e-3
        assert tr["outcome"] is not None and tr["outcome"]["termination"] in ("Checkmate", "Stalemate")
    eng.close()

    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 16)
    seeds = list(range(100, 116))
    kw = dict(rollout_num=30, num_steps=16, cpuct=2.5, temperature_switch=4, with_noise=True)
    many, _ = scb200.game_selfplay_many(eng, seeds, **kw)
    for s, tr in zip(seeds, many):
        assert tr == scb200.game_selfplay(eng, seed=s, **kw)
    eng.close()


def test_lifecycle(blob):
    import scb200

    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 8)
    pos, moves, off = scb200.random_positions(2, seed=1)
    ref = eng.eval(pos, moves, off)
    ev = scb200.Evaluator(eng, 4)
    rc = scb200.load_library().sc_set_roots(eng.handle, 0, None, None)
    assert rc == SC_E_STATE and "evaluator" in scb200.last_error()
    with pytest.raises(scb200.SCError, match=r"\(-5\)"):
        eng.eval(pos, moves, off)
    with pytest.raises(scb200.SCError, match=r"\(-5\)"):
        scb200.Evaluator(eng, 4)
    ev.set_root(0, [])
    assert ev.predict(0, [])[1] == 20
    ev.close()  # (callers still queued then get SC_E_STATE: csrc/host/tsan_main.cpp checks that without a GPU)
    assert ev.predict(0, [], check=False)[0] == SC_E_STATE
    got = eng.eval(pos, moves, off)  # the engine works again
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    eng.close()
