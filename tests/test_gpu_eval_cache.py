"""The evaluation cache (sc_set_eval_cache): sc_predict, sc_predict_stack, sc_predict_path and the batching evaluator on a
cached engine return exactly what an engine without a cache returns -- outputs, statuses and messages -- and the
counts say how each leaf was answered.  Every check compares a cached engine against an uncached engine of the same
blob, bit for bit."""
import json
import os

import numpy as np
import pytest

from test_gpu_evaluator import _reference, _run_threads, _same, leaves  # noqa: F401  (fixture)
from test_gpu_predict import OVERFLOW_BOARDS, _raw_predict
from test_gpu_predict_path import _flat, _raw_predict_path, _random_games
from test_gpu_predict_path import _rejections as _path_rejections
from test_gpu_predict_stack import FOOLS_MATE, SMOTHERED_MATE, STALEMATE
from test_gpu_predict_stack import _rejections as _stack_rejections

pytestmark = pytest.mark.gpu

MODES = ("SC_MODE_FP32", "SC_MODE_BF16", "SC_MODE_FP32_FFMA", "SC_MODE_FP16", "SC_MODE_FP8")
SIZES = (1, 37, 129, 2048)
BIG = 1 << 18  # 65536 buckets: the pools below never fill one, so nothing is evicted
SC_E_INVAL, SC_E_STATE = -1, -5
# kernels of a call whose leaves all hit: the cache's probe and finish kernels (+ the replay of sc_predict_stack/_path)
ALL_HIT_LAUNCHES = {"predict": 2, "stack": 3, "path": 3}


@pytest.fixture(scope="module")
def blob(tmp_path_factory):
    import net
    import scb200

    p = str(tmp_path_factory.mktemp("eval_cache") / "w.scw")
    scb200.write_blob(net.perturb_norm_params(net.init_state_dict(2, 7), 1234), p)
    return p


def _ep(stack, pos):
    """python-chess ep_square after `stack`: the skipped square after a pawn's double push"""
    if not stack:
        return -1
    f, t, _ = stack[-1]
    pawn = (int(pos["slot"][0][0]) >> t) & 1
    return (f + t) // 2 if pawn and abs(t - f) == 16 else -1


@pytest.fixture(scope="module")
def pool(blob):
    """distinct leaves (no two share the packed row and the ep byte), in shuffled order, each as a root index and a
    path (roots: every 30th prefix of 48 random games), its whole stack, and its packed position and ep square"""
    import scb200

    games = _random_games(48, 300, seed=5)
    roots, root_of = [], {}
    for g, game in enumerate(games):
        for a in range(0, len(game) + 1, 30):
            root_of[(g, a)] = len(roots)
            roots.append(game[:a])
    cand = [(root_of[(g, L - L % 30)], game[L - L % 30 : L], game[:L]) for g, game in enumerate(games)
            for L in range(len(game) + 1)]
    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 2048)
    keys, out = set(), []
    for b in range(0, len(cand), 2048):
        chunk = cand[b : b + 2048]
        pos = eng.predict_stack([c[2] for c in chunk], positions=True)[4]
        for c, p in zip(chunk, pos):
            ep = _ep(c[2], p)
            k = p.tobytes() + bytes([ep & 0xFF])
            if k not in keys:
                keys.add(k)
                out.append((c[0], c[1], c[2], p, ep))
    eng.close()
    order = np.random.RandomState(3).permutation(len(out))
    return roots, [out[i] for i in order]


GUARD_ROWS = 2


def _call(e, kind, roots, leaves):
    """one call of `kind` on `leaves` (pool entries): (rc, moves, counts, priors, values, positions or None).  The
    output arrays have GUARD_ROWS canary rows after row n, which the call must leave as they are"""
    import scb200

    n = len(leaves)
    buf = (np.full((n + GUARD_ROWS, scb200.SC_MAX_MOVES), 0xAB, dtype=np.uint32).view(scb200.MOVE_DTYPE),
           np.full(n + GUARD_ROWS, -7, dtype=np.int32), np.full((n + GUARD_ROWS, scb200.SC_MAX_MOVES), 7.0, dtype=np.float32),
           np.full(n + GUARD_ROWS, 7.0, dtype=np.float32))
    if kind == "predict":
        pos = np.array([lv[3] for lv in leaves], dtype=scb200.POSITION_DTYPE)
        ep = np.array([lv[4] for lv in leaves], dtype=np.int8)
        res = e.predict(pos, ep, out=buf, check=False) + (None,)
    elif kind == "stack":
        res = e.predict_stack([lv[2] for lv in leaves], out=buf, positions=True, check=False)
    else:
        res = e.predict_path([lv[0] for lv in leaves], [lv[1] for lv in leaves], out=buf, positions=True, check=False)
    moves, cnt, priors, vals = buf
    assert (moves[n:].view(np.uint32) == 0xAB).all() and (cnt[n:] == -7).all(), "written past row n"
    assert (priors[n:] == 7.0).all() and (vals[n:] == 7.0).all(), "written past row n"
    return res


def _assert_equal(got, exp, what):
    rc, moves, cnt, priors, vals, pos = got
    erc, emoves, ecnt, epriors, evals, epos = exp
    assert rc == erc and np.array_equal(cnt, ecnt), what
    for i in range(len(cnt)):
        c = int(cnt[i])
        assert np.array_equal(moves[i, :c].view(np.uint32), emoves[i, :c].view(np.uint32)), (what, i)
        assert np.array_equal(priors[i, :c].view(np.uint32), epriors[i, :c].view(np.uint32)), (what, i)
    assert np.array_equal(vals.view(np.uint32), evals.view(np.uint32)), what
    if pos is not None:
        assert pos.tobytes() == epos.tobytes(), what


def _delta(e, before):
    now = e.eval_cache_stats()
    return {k: now[k] - before[k] for k in ("lookups", "hits", "duplicates", "inserts", "evictions")}


def _counts(lookups, hits=0, duplicates=0, inserts=0, evictions=0):
    return dict(lookups=lookups, hits=hits, duplicates=duplicates, inserts=inserts, evictions=evictions)


@pytest.mark.parametrize("mode", MODES)
def test_outputs_and_counts_equal_uncached(blob, pool, mode):
    """all misses, the same call again (all hits, no network), half old and half new leaves shuffled, and k leaves
    three times each on a fresh table, at n = 1, 37, 129, 2048, through the three entry points"""
    import scb200

    roots, lv = pool
    ref = scb200.Engine(blob, 0, getattr(scb200, mode), 2048)
    e = scb200.Engine(blob, 0, getattr(scb200, mode), 2048)
    rng = np.random.RandomState(1)
    try:
        for kind in ("predict", "stack", "path"):
            if kind == "path":
                ref.set_roots(roots)
                e.set_roots(roots)
            for n in SIZES:
                e.set_eval_cache(BIG)
                assert e.eval_cache_stats() == dict(entries=BIG, **_counts(0))
                old, new = lv[:n], lv[n : 2 * n - n // 2]
                half = old[: n // 2] + new
                half = [half[i] for i in rng.permutation(len(half))]
                k = max(1, n // 3)
                trip = lv[2 * n : 2 * n + k] * 3
                trip = [trip[i] for i in rng.permutation(len(trip))]
                for name, leaves, exp, fresh in (
                    ("first", old, _counts(n, inserts=n), False),
                    ("again", old, _counts(n, hits=n), False),
                    ("half", half, _counts(n, hits=n // 2, inserts=n - n // 2), False),
                    ("thrice", trip, _counts(3 * k, duplicates=2 * k, inserts=k), True),
                ):
                    if fresh:
                        e.set_eval_cache(BIG)
                    before, launches = e.eval_cache_stats(), e.launch_count()
                    got = _call(e, kind, roots, leaves)
                    assert _delta(e, before) == exp, (mode, kind, n, name)
                    if name == "again":
                        assert e.launch_count() - launches == ALL_HIT_LAUNCHES[kind], (mode, kind, n)
                    _assert_equal(got, _call(ref, kind, roots, leaves), (mode, kind, n, name))
                    assert got[0] == 0
    finally:
        e.close()
        ref.close()


def test_one_bucket_table(blob, pool):
    """a table of one bucket (4 entries) that every key competes for"""
    import scb200

    roots, lv = pool
    ref = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 1024)
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 1024)
    try:
        e.set_eval_cache(1)
        assert e.eval_cache_stats()["entries"] == 4
        # 300 distinct leaves in calls of 1..9 rows, each call repeating some leaves of the last two calls
        rng = np.random.RandomState(2)
        seen, nxt, total = [], 0, 0
        while nxt < 300:
            m = int(rng.randint(1, 10))
            rows = lv[nxt : nxt + m] + [seen[i] for i in rng.randint(0, len(seen), size=int(rng.randint(0, 4)))] if seen \
                else lv[nxt : nxt + m]
            nxt += m
            seen = (seen + lv[nxt - m : nxt])[-12:]
            rows = [rows[i] for i in rng.permutation(len(rows))]
            for kind in ("predict", "stack"):
                _assert_equal(_call(e, kind, roots, rows), _call(ref, kind, roots, rows), ("interleaved", nxt, kind))
                total += len(rows)
        st = e.eval_cache_stats()
        print("one bucket, interleaved:", st)
        assert st["lookups"] == total and st["evictions"] > 0 and st["hits"] > 0
        assert st["inserts"] - st["evictions"] <= 4

        # hits and new leaves in one bucket: the hits' entries are kept, the new results are not stored
        e.set_eval_cache(1)
        a, b = lv[400:404], lv[404:408]
        _call(e, "predict", roots, a)
        before = e.eval_cache_stats()
        rows = a + b
        _assert_equal(_call(e, "predict", roots, rows), _call(ref, "predict", roots, rows), "shared bucket")
        assert _delta(e, before) == _counts(8, hits=4)
        # two hits pin two ways: two of the four new leaves replace the other two entries
        before = e.eval_cache_stats()
        rows = b + a[:2]
        _assert_equal(_call(e, "predict", roots, rows), _call(ref, "predict", roots, rows), "shared bucket 2")
        assert _delta(e, before) == _counts(6, hits=2, inserts=2, evictions=2)
        before = e.eval_cache_stats()
        _assert_equal(_call(e, "predict", roots, a), _call(ref, "predict", roots, a), "shared bucket 3")
        assert _delta(e, before)["hits"] == 2

        # random bytes next to real leaves, twice (miss, then whatever the bucket kept); nothing written past row n
        rng = np.random.RandomState(9)
        n = 256
        pos = rng.randint(0, 256, size=n * scb200.POSITION_DTYPE.itemsize, dtype=np.uint8).view(scb200.POSITION_DTYPE)
        ep = rng.choice([-1] + list(range(16, 24)) + list(range(40, 48)), size=n).astype(np.int8)
        pos[0::2] = np.array([x[3] for x in lv[500 : 500 + n // 2]], dtype=scb200.POSITION_DTYPE)
        ep[0::2] = [x[4] for x in lv[500 : 500 + n // 2]]
        pos[::3] = pos[0]  # and duplicates of one leaf
        ep[::3] = ep[0]
        for rep in range(2):
            got, exp = _raw_predict(e, pos, ep), _raw_predict(ref, pos, ep)
            _assert_equal(got + (None,), exp + (None,), ("random positions", rep))
        paths = [list(x[1]) for x in lv[600:664]]
        root = [x[0] for x in lv[600:664]]
        for i in range(1, 64, 2):  # move fields the host accepts, mostly rejected by the replay
            paths[i] = [(int(f), int(t), int(p)) for f, t, p in zip(rng.randint(0, 64, 5), rng.randint(0, 64, 5),
                                                                    rng.choice([0, 2, 3, 4, 5], 5))]
        e.set_roots(roots)
        ref.set_roots(roots)
        for rep in range(2):
            rc, msg, got = _raw_predict_path(e, root, *_flat(paths))
            erc, emsg, exp = _raw_predict_path(ref, root, *_flat(paths))
            assert msg == emsg
            _assert_equal((rc,) + got, (erc,) + exp, ("random paths", rep))
        assert e.eval_cache_stats()["evictions"] > 0
    finally:
        e.close()
        ref.close()


def test_power_of_two_table_uses_every_bucket(blob, pool):
    """a table of 1024 entries (256 buckets of 4) filled with 1024 distinct leaves in one call keeps about 80 % of them
    (the share a 4-way table with 4 keys per bucket on average holds); a table reaching only half its buckets would keep
    at most 512.  The same call again hits exactly the stored ones"""
    import scb200

    roots, lv = pool
    ref = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 1024)
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 1024)
    try:
        for entries in (1024, 1000):  # a power of two, and 250 buckets
            e.set_eval_cache(entries)
            rows = lv[:entries]
            _assert_equal(_call(e, "stack", roots, rows), _call(ref, "stack", roots, rows), ("fill", entries))
            st = e.eval_cache_stats()
            print("fill", entries, st)
            assert st["evictions"] == 0 and 0.7 * entries < st["inserts"] <= entries
            _assert_equal(_call(e, "stack", roots, rows), _call(ref, "stack", roots, rows), ("again", entries))
            assert e.eval_cache_stats()["hits"] == st["inserts"]
    finally:
        e.close()
        ref.close()


def test_terminal_and_rejected_leaves(blob):
    import scb200

    L = scb200.load_library()
    ref = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 256)
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 256)
    try:
        e.set_eval_cache(4096)
        stacks = [FOOLS_MATE[0], SMOTHERED_MATE[0], STALEMATE[0], []]
        for rep in range(2):  # miss, then hit
            got = e.predict_stack(stacks, positions=True, check=False)
            _assert_equal(got, ref.predict_stack(stacks, positions=True, check=False), ("terminal", rep))
            assert got[2].tolist() == [0, 0, 0, 20]
            assert got[4].tolist()[:3] == [FOOLS_MATE[1], SMOTHERED_MATE[1], STALEMATE[1]]
        assert e.eval_cache_stats()["hits"] == 4
        # more than 256 pseudo-legal moves: the call fails with the same message when the leaf hits
        bad = np.zeros(1, dtype=scb200.POSITION_DTYPE)
        for k, b in enumerate(OVERFLOW_BOARDS):
            bad["slot"][0, 0, k] = b
        bad["slot"][0, 0, 6] = sum(OVERFLOW_BOARDS)
        bad["meta"][0] = (1, 1, 0, 0, 0, 0, 0)
        bad["n_hist"][0] = 1
        start = e.predict_stack([[]], positions=True)[4]
        trio = np.concatenate([start, bad, start])
        for batch in (trio, np.concatenate([trio] * 60)):
            for rep in range(2):
                got = _raw_predict(e, batch, None)
                msg = L.sc_last_error().decode()
                exp = _raw_predict(ref, batch, None)
                assert msg == L.sc_last_error().decode() and "leaf 1 has more than 256" in msg
                _assert_equal(got + (None,), exp + (None,), ("overflow", len(batch), rep))
        # replay-time rejections of stacks, paths and roots
        for stack, ply, words in _stack_rejections():
            stacks = [[], _uci_d4(), stack]
            for rep in range(2):
                got = e.predict_stack(stacks, positions=True, check=False)
                msg = L.sc_last_error().decode()
                exp = ref.predict_stack(stacks, positions=True, check=False)
                assert msg == L.sc_last_error().decode() and f"leaf 2, ply {ply}" in msg and words in msg
                _assert_equal(got, exp, (stack, rep))
        for stack, ply, words in _path_rejections():
            roots, paths = [[], stack[:1], _uci_d4()], [[], stack[1:], []]
            for eng in (e, ref):
                eng.set_roots(roots)
            for rep in range(2):
                rc, msg, got = _raw_predict_path(e, [0, 1, 2], *_flat(paths))
                erc, emsg, exp = _raw_predict_path(ref, [0, 1, 2], *_flat(paths))
                assert rc == erc == SC_E_INVAL and msg == emsg
                _assert_equal((rc,) + got, (erc,) + exp, (stack, rep))
            flat, off = _flat([stack])
            for eng in (e, ref):
                rc = L.sc_set_roots(eng.handle, 1, flat.ctypes.data, off.ctypes.data)
                assert rc == SC_E_INVAL and f"root 0, ply {ply}" in L.sc_last_error().decode()
    finally:
        e.close()
        ref.close()


def _uci_d4():
    return [(11, 27, 0)]


def test_evaluator_threads_equal_predict_stack(blob, leaves):  # noqa: F811
    """64 threads, every leaf twice (the second round hits), against predict_stack on an uncached engine"""
    import scb200

    roots, specs = leaves
    ref_eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 512)
    ref = _reference(ref_eng, roots, specs)
    ref_eng.close()
    eng = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 512)
    eng.set_eval_cache(1 << 14)
    ev = scb200.Evaluator(eng, len(roots))
    for g, r in enumerate(roots):
        ev.set_root(g, r)
    got = [None] * (2 * len(specs))
    stats_seen = []

    def work(t):
        for i in range(t, len(got), 64):
            g, p = specs[i % len(specs)]
            got[i] = ev.predict(g, p, positions=True, check=False)
        if t == 0:
            stats_seen.append(eng.eval_cache_stats())  # readable while the evaluator runs

    _run_threads(64, work)
    for i, r in enumerate(got):
        _same(r, ref[i % len(specs)])
    st = eng.eval_cache_stats()
    print("evaluator, 64 threads:", st, ev.stats())
    assert stats_seen and st["lookups"] == len(got) and st["hits"] + st["duplicates"] >= len(specs)
    ev.close()
    eng.close()


def test_selfplay_many_traces_equal_uncached(blob):
    """16 games with root noise and a temperature switch at ply 4: the cached engine plays the uncached engine's games"""
    import scb200

    kw = dict(rollout_num=30, num_steps=16, cpuct=2.5, temperature_switch=4, with_noise=True, epsilon=0.15)
    seeds = list(range(200, 216))
    ref = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 16)
    exp, _ = scb200.game_selfplay_many(ref, seeds, **kw)
    ref.close()
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 16)
    e.set_eval_cache(1 << 16)
    got, counts = scb200.game_selfplay_many(e, seeds, **kw)
    st = e.eval_cache_stats()
    print("16 games:", st, counts)
    assert got == exp
    assert st["hits"] > 0 and st["lookups"] == counts["leaves"]
    e.close()


def test_golden_game_on_a_cached_engine(tmp_path):
    """configs[0] (fp32, seed-0 19-block net, 20 rollouts, no noise): the golden game, with most leaves from the cache"""
    import scb200

    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "search_cfg1.json")))
    cfg = gold["config"]
    blob19 = str(tmp_path / "seed0.scw")
    scb200.write_blob(scb200.random_init_state_dict(cfg["n_res_blocks"], 0), blob19)
    eng = scb200.Engine(blob19, 0, scb200.SC_MODE_FP32, 2)
    eng.set_eval_cache(1 << 16)
    traces, counts = scb200.game_selfplay_many(eng, [0, 0], rollout_num=cfg["rollout_num"], num_steps=cfg["num_steps"],
                                               cpuct=cfg["cpuct"])
    st = eng.eval_cache_stats()
    print("golden game, cached:", st, counts)
    for tr in traces:
        assert len(tr["steps"]) == len(gold["steps"])
        for (mv, q, ch), r in zip(tr["steps"], gold["steps"]):
            assert mv == r["move"]
            assert [(c[0], c[1]) for c in ch] == [(c[0], c[1]) for c in r["children"]]
            assert max(abs(c[2] - x[2]) for c, x in zip(ch, r["children"])) < 1e-3
    assert st["hits"] > 0
    eng.close()


def test_api(blob, pool):
    import scb200

    L = scb200.load_library()
    roots, lv = pool
    e = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 64)
    ref = scb200.Engine(blob, 0, scb200.SC_MODE_BF16, 64)
    try:
        assert e.eval_cache_stats() == dict(entries=0, **_counts(0))
        for bad in (-1, scb200.SC_MAX_CACHE_ENTRIES + 1):
            assert L.sc_set_eval_cache(e.handle, bad) == SC_E_INVAL
        assert L.sc_set_eval_cache(e.handle, scb200.SC_MAX_CACHE_ENTRIES) == 0
        assert e.eval_cache_stats()["entries"] == scb200.SC_MAX_CACHE_ENTRIES
        e.set_eval_cache(10)
        assert e.eval_cache_stats()["entries"] == 12  # whole buckets of 4
        rows = lv[:3]
        _call(e, "stack", roots, rows)
        assert e.eval_cache_stats()["hits"] == 0
        _call(e, "stack", roots, rows)
        assert e.eval_cache_stats()["hits"] == 3
        e.set_eval_cache(100)  # a new table is empty
        before = e.eval_cache_stats()
        assert before == dict(entries=100, **_counts(0))
        _assert_equal(_call(e, "stack", roots, rows), _call(ref, "stack", roots, rows), "resized")
        assert _delta(e, before) == _counts(3, inserts=3)
        # an evaluator owns the engine: SC_E_STATE, stats still readable; after it is gone the call works
        ev = scb200.Evaluator(e, 2)
        ev.set_root(0, [])
        ev.predict(0, [])
        assert L.sc_set_eval_cache(e.handle, 16) == SC_E_STATE and "evaluator" in scb200.last_error()
        assert e.eval_cache_stats()["lookups"] == 4
        ev.close()
        e.set_eval_cache(16)
        # 0 turns the cache off
        e.set_eval_cache(0)
        assert e.eval_cache_stats() == dict(entries=0, **_counts(0))
        for _ in range(2):
            _assert_equal(_call(e, "stack", roots, rows), _call(ref, "stack", roots, rows), "off")
        assert e.eval_cache_stats()["lookups"] == 0
    finally:
        e.close()
        ref.close()
