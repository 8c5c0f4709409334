"""bench.py's host-side pieces that need no GPU: the config object both arms print, the reference arm
(compiled reference search, oracle/_ref, driving a network callback from host threads in both feeding
modes) on a tiny CPU network, and the shape of its result object."""
import argparse

import pytest
import torch

import bench
from tests import oracles


def test_both_arms_print_the_same_config_object():
    a = argparse.Namespace(games=4096, nn_batch=256, parts=2, opening_plies=16)
    for world in (1, 2, 8):
        ours = bench.selfplay_config(a, world, "net")
        ref = bench.selfplay_config(a, world, "net")
        assert ours == ref and ours["games_per_gpu"] == 4096 // world
        assert ("configs[2]" in ours["workload"]) == (world == 1) and ("configs[3]" in ours["workload"]) == (world > 1)


def test_defaults_are_the_self_play_workload(monkeypatch):
    seen = {}
    monkeypatch.setattr(bench, "run_selfplay", lambda args: seen.setdefault("ours", args) and 0)
    monkeypatch.setattr(bench, "run_reference_selfplay", lambda args: seen.setdefault("ref", args) and 0)
    monkeypatch.setattr(bench.os, "dup2", lambda a, b: None)
    monkeypatch.setattr("sys.argv", ["bench.py"])
    bench.main()
    monkeypatch.setattr("sys.argv", ["bench.py", "--impl", "reference", "--gpus", "2"])
    bench.main()
    assert seen["ours"].workload == "selfplay" and seen["ours"].games == 4096 and seen["ours"].steps == 20
    assert seen["ours"].warmup >= 3 and seen["ref"].gpus == 2


@pytest.mark.timeout(600)
def test_reference_arm_on_a_tiny_cpu_network():
    """the --impl reference arm end to end, minus the GPU: 800-rollout moves in 80-rollout slices on the
    compiled reference search, one call per wave and batched through the collector"""
    if not oracles.have_ref(19):
        pytest.skip("oracle/_ref not built")
    from elf_b200.model import FusedActor, PolicyValueNet

    torch.manual_seed(0)
    fa = FusedActor(PolicyValueNet(19, num_block=1, dim=8).eval(), batchsize=256, dtype=torch.float32, cuda_graph=False)
    r = bench.ref_selfplay(fa, torch.device("cpu"), steps=2, warmup=1)
    assert r["kind"] == "reference" and r["unit"] == "moves/s" and r["value"] > 0 and r["cores"] >= 1
    assert set(r["modes"]) == {"one_call_per_wave", "batched"} and r["mode"] in r["modes"]
    for m in r["modes"].values():
        assert m["value"] > 0 and m["nn_positions_per_s"] > 0
    assert r["value"] == max(m["value"] for m in r["modes"].values())


def test_steps_sets_the_timed_steps_of_both_workloads(monkeypatch):
    seen = []
    monkeypatch.setattr(bench, "run_selfplay", lambda args: seen.append(args) and 0)
    monkeypatch.setattr(bench, "run_playout", lambda args: seen.append(args) and 0)
    monkeypatch.setattr(bench.os, "dup2", lambda a, b: None)
    for argv, steps in ((["--workload", "playout", "--steps", "20"], 20), (["--workload", "playout"], 30),
                        (["--steps", "7"], 7), (["--steps", "30"], 30)):
        monkeypatch.setattr("sys.argv", ["bench.py"] + argv)
        bench.main()
        assert seen[-1].steps == steps, argv
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "3", "--dump-outputs", "d"])
    bench.main()
    assert seen[-1].dump_outputs == "d" and seen[-1].steps == 3


def test_dump_outputs_writes_float_arrays_one_row_per_game(tmp_path, monkeypatch):
    import numpy as np

    G = 50
    rng = np.random.default_rng(1)
    arrays = {"visits": rng.integers(0, 800, (G, 82)).astype(np.int32), "q": rng.random(G).astype(np.float32),
              "hash": rng.integers(0, 2**63, G, dtype=np.int64).astype(np.uint64) * np.uint64(2) + np.uint64(1)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    got = {p.stem: np.load(p) for p in (tmp_path / "all").iterdir()}
    assert set(got) == {"visits", "q", "hash_hi", "hash_lo", "game_index"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert (got["visits"] == arrays["visits"]).all() and (got["q"] == arrays["q"]).all()
    h = (got["hash_hi"].astype(np.uint64) << np.uint64(32)) | got["hash_lo"].astype(np.uint64)
    assert (h == arrays["hash"]).all() and (got["game_index"] == np.arange(G)).all()
    # above the size limit: the same seeded sample of games, in every array and from run to run
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 20 * (82 * 8 + 4 + 3 * 8))
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    s1, s2 = ({p.stem: np.load(p) for p in (tmp_path / d).iterdir()} for d in ("s1", "s2"))
    keep = s1["game_index"].astype(int)
    assert len(keep) == 20 and (np.diff(keep) > 0).all() and all((s1[k] == s2[k]).all() for k in s1)
    assert (s1["visits"] == arrays["visits"][keep]).all() and (s1["q"] == arrays["q"][keep]).all()
