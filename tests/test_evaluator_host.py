"""CPU test of the batching evaluator's queue (sc_game_selfplay_many with the position-hash stand-in): games played on
many threads through one evaluator equal the same seeds played one at a time, and the passes carry several leaves."""


def test_game_selfplay_many_hash_equals_games_alone():
    import scb200

    seeds = list(range(40, 72))
    kw = dict(rollout_num=10, num_steps=24, cpuct=2.5, temperature_switch=5, with_noise=True, evaluator="hash")
    traces, counts = scb200.game_selfplay_many(None, seeds, **kw)
    assert counts["largest_batch"] > 1 and counts["passes"] < counts["leaves"]
    assert counts["root_updates"] >= sum(len(t["steps"]) for t in traces)
    for s, tr in zip(seeds, traces):
        assert tr == scb200.game_selfplay(None, seed=s, **kw)
