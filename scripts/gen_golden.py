#!/usr/bin/env python
"""Generate tests/golden/*.json from the compiled UNMODIFIED reference (oracle/_ref).

Run in the CPU container (needs /root/reference to have been compiled by `make -C oracle ref`).
The fixtures are committed; the GPU box only reads them.
  playouts_{19,9}.json : for seed 2026, game ids 0..63 -> plies, position checksum, final tt
                         score; for game ids 0,1 the full move list, per-ply hash and captures.
  positions_{19,9}.json: a few mid-game positions reached by those move lists, with the
                         reference's legal mask, true-eye masks, tt score, evaluate(7.5), info
                         words and AGZ feature planes (as indices of the ones) under several D4.
"""
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import oracles  # noqa: E402

SEED = 2026


def gen(n):
    L = oracles.load_ref(n)
    maxp = 2 * n * n
    games = []
    for gid in range(64):
        chk = ctypes.c_uint64()
        sc = ctypes.c_int32()
        moves = np.zeros(maxp, np.int32)
        hashes = np.zeros(maxp, np.uint64)
        caps = np.zeros(2 * maxp, np.int32)
        t = L.ref_playout(SEED, gid, maxp, moves.ctypes.data, hashes.ctypes.data, caps.ctypes.data,
                          ctypes.byref(chk), ctypes.byref(sc))
        e = {"game_id": gid, "plies": int(t), "chk": f"{chk.value:016x}", "score": int(sc.value)}
        if gid < 2:
            e["moves"] = moves[:t].tolist()
            e["hashes"] = [f"{int(h):016x}" for h in hashes[:t]]
            e["caps"] = caps[: 2 * t].reshape(-1, 2).tolist()
        games.append(e)
    with open(os.path.join(ROOT, "tests", "golden", f"playouts_{n}.json"), "w") as f:
        json.dump({"board_size": n, "seed": SEED, "games": games}, f)

    positions = []
    for gid in range(2):
        r = oracles.Ref(n)
        mv = games[gid]["moves"]
        stops = sorted(set([3, 9, len(mv) // 3, len(mv) // 2, (3 * len(mv)) // 4, len(mv) - 2, len(mv)]))
        for t, a in enumerate(mv, start=1):
            assert r.forward(a)
            if t in stops:
                info = r.info()
                feats = {}
                for d4 in (0, 3, 5, 6):
                    feats[str(d4)] = np.flatnonzero(r.features(d4).reshape(-1)).tolist()
                positions.append({
                    "game_id": gid, "after_ply": t, "hash": f"{r.hash():016x}", "info": info.tolist(),
                    "stones": r.stones().tolist(), "legal": r.legal().tolist(),
                    "eyes_black": np.flatnonzero(r.true_eyes(1)).tolist(),
                    "eyes_white": np.flatnonzero(r.true_eyes(2)).tolist(),
                    "tt_score": r.tt_score(), "evaluate_7_5": r.evaluate(7.5), "features_ones": feats,
                })
    with open(os.path.join(ROOT, "tests", "golden", f"positions_{n}.json"), "w") as f:
        json.dump({"board_size": n, "seed": SEED, "positions": positions}, f)


if __name__ == "__main__":
    for n in (19, 9):
        gen(n)
        print("golden fixtures written for", n)


def gen_mcts():
    """tests/golden/mcts_<scenario>.json: root visit counts of the compiled reference search."""
    from tests.test_mcts_oracle_vs_ref import SCENARIOS, ref_mcts, run_search

    for name, sc in sorted(SCENARIOS.items()):
        n = sc["n"]
        res, evals = run_search(sc, lambda: oracles.Ref(n), lambda: ref_mcts(sc))
        steps = []
        for r in res:
            v = r["visits"]
            steps.append({"best_action": r["best_action"], "total_visits": r["total_visits"],
                          "visits": {str(int(a)): int(v[a]) for a in np.flatnonzero(v >= 0)}})
        with open(os.path.join(ROOT, "tests", "golden", f"mcts_{name}.json"), "w") as f:
            json.dump({"scenario": name, "num_evals": evals, "steps": steps}, f)
        print("golden mcts fixture", name)


def gen_scale_sample():
    """tests/golden/mcts_19_scale_sample.json: the compiled reference search's root-table records (move,
    total visits, root value, digest of visits and priors) of the 64 sampled games of
    tests/test_gpu_search_at_scale.py.  Each game's opening comes from a generator of its own, so only the
    sampled games are searched."""
    from tests import test_gpu_search_at_scale as S

    games = S.sample_games(4096)
    d = {"seed": S.SEED, "opts": S.OPTS, "games": games.tolist(), "tables": S.reference_records(games)}
    with open(S.GOLD, "w") as f:
        json.dump(d, f)
    print("golden mcts fixture 19_scale_sample")


if __name__ == "__main__" and (len(sys.argv) == 1 or "mcts" in sys.argv):
    gen_mcts()
if __name__ == "__main__" and (len(sys.argv) == 1 or "scale" in sys.argv):
    gen_scale_sample()
