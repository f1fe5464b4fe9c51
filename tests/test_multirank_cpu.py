"""world_size-2 gloo test of the N>1 host logic (game sharding + counter reduction), on CPU with the
driver's position-hash evaluator standing in for the device."""
import os
import socket
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_arithmetic():
    from scb200 import shard

    for n in (0, 1, 7, 500, 16384):
        for w in (1, 2, 4, 8):
            assert sum(shard.games_for_rank(n, r, w) for r in range(w)) == n
            ids = sorted(i for r in range(w) for i in shard.game_ids_for_rank(n, r, w))
            assert ids == list(range(n))
    assert shard.rank_seed(5, 0) != shard.rank_seed(5, 1)


def test_two_ranks_gloo(tmp_path):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    script = tmp_path / "worker.py"
    script.write_text(textwrap.dedent(f"""
        import os, sys, json
        sys.path.insert(0, {ROOT!r}); sys.path.insert(0, os.path.join({ROOT!r}, "smart-chess-rust_b200"))
        import torch.distributed as dist
        import scb200
        from scb200 import shard
        dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
        rank, world = dist.get_rank(), dist.get_world_size()
        n_games = 7
        mine = shard.games_for_rank(n_games, rank, world)
        sp = scb200.SelfPlay(None, n_trees=4, rollout_num=12, num_steps=10, cpuct=2.5, with_noise=True,
                             temperature_switch=4, evaluator="hash", seed=shard.rank_seed(3, rank), keep_traces=True)
        st = sp.run(max_games=mine)
        first = sp.trace(0)["steps"][0][0]
        tot = shard.reduce_stats(st, dist)
        if rank == 0:
            print(json.dumps({{"tot": tot, "mine": mine, "local": st["games_finished"]}}))
        dist.barrier()
        dist.destroy_process_group()
    """))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=120) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    import json

    d = json.loads(outs[0][0].strip().splitlines()[-1])
    assert d["mine"] == 4 and d["local"] == 4
    assert d["tot"]["games_finished"] == 7
    assert d["tot"]["moves"] == 7 * 10
    assert d["tot"]["rollouts"] == 7 * 10 * 12


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the oracle port on the host cores) needs no GPU: one JSON line with the keys the
    driver reads, `config` identical in shape to the GPU arm's, the real step size when it fits the time budget."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--leaves", "64"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "leaf_evals_per_s" and d["unit"] == "leaf evals/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    assert d["config"]["leaves_per_step"] == 64 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["leaves_per_step_run"] == 64
    assert cb["batch1_value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "leaf evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_dump_outputs_refused_on_the_reference_arm(tmp_path):
    """The reference arm keeps no outputs: --dump-outputs there is an error, not an empty directory."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                        str(tmp_path / "d")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


def test_bench_dump_outputs_sample_stays_under_the_cap_and_splits_by_leaf(tmp_path, monkeypatch):
    import numpy as np

    import bench

    rng = np.random.default_rng(1)
    off = np.concatenate([[0], np.cumsum(rng.integers(0, 60, 3000))]).astype(np.int32)
    pri, val = rng.random(off[-1]).astype(np.float32), rng.random(3000).astype(np.float32)
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    for world, rank in ((1, 0), (2, 1)):
        d = tmp_path / str(world)
        bench.dump_outputs(str(d), pri, val, off, rank, world)
        assert sum(f.stat().st_size for f in d.iterdir()) <= 200_000 // world
        s = "" if world == 1 else "_rank1"
        p, v, lv, o = (np.load(d / f"{n}{s}.npy") for n in ("priors", "values", "leaves", "offsets"))
        lv, o = lv.astype(np.int64), o.astype(np.int64)
        assert 0 < len(lv) < 3000 and (np.diff(lv) > 0).all() and np.array_equal(v, val[lv]) and o[-1] == len(p)
        for k, i in enumerate(lv):
            assert np.array_equal(p[o[k]:o[k + 1]], pri[off[i]:off[i + 1]])
