"""Pin the C restatement of the tree search (oracle/mcts_oracle.c) against the compiled UNMODIFIED
reference search (MCTSAI_T / TreeSearchT / MCTSActor logic through oracle/_ref): identical root
edge sets, visit counts, reward sums, priors, values and number of network evaluations, move after
move with a persistent tree.  Also against the committed golden vectors (no reference needed)."""
import json
import os

import numpy as np
import pytest

from tests import oracles

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

SCENARIOS = {
    "19_persistent_b8": dict(n=19, G=3, moves=5, open_plies=6,
                             opts=dict(num_rollouts=200, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1, c_puct=1.5)),
    "19_fresh_b1": dict(n=19, G=2, moves=3, open_plies=30,
                        opts=dict(num_rollouts=96, num_rollouts_per_batch=1, virtual_loss=0, persistent_tree=0, c_puct=0.85)),
    "19_midgame_800": dict(n=19, G=2, moves=2, open_plies=60,
                           opts=dict(num_rollouts=800, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1, c_puct=1.5)),
    "9_endgame": dict(n=9, G=6, moves=12, open_plies=60,
                      opts=dict(num_rollouts=160, num_rollouts_per_batch=4, virtual_loss=2, persistent_tree=1, c_puct=1.5)),
    "9_root_uqz_noprior": dict(n=9, G=3, moves=6, open_plies=30,
                               opts=dict(num_rollouts=80, num_rollouts_per_batch=5, virtual_loss=3, persistent_tree=1, c_puct=1.0,
                                         root_unexplored_q_zero=1)),
    "9_uqz_pass": dict(n=9, G=4, moves=10, open_plies=50,
                       opts=dict(num_rollouts=120, num_rollouts_per_batch=6, virtual_loss=1, persistent_tree=1, c_puct=2.0,
                                 unexplored_q_zero=1, ply_pass_enabled=40, remove_pass_if_dangerous=0)),
    # exact PUCT-score ties, which the reference resolves in the iteration order of its unordered_map
    # (NodeT::UCT, tree_search_node.h:361-397): without the prior term every unvisited edge ties ...
    "9_noprior_ties": dict(n=9, G=3, moves=5, open_plies=40,
                           opts=dict(num_rollouts=60, num_rollouts_per_batch=6, virtual_loss=1, persistent_tree=1, c_puct=1.5,
                                     use_prior=0)),
    # ... and with it, priors small enough that c_puct * P * sqrt(n) vanishes under the rounding of q tie as
    # well (late positions; the fixed openings were found by scripts/emu_fuzz.py)
    "9_rounding_ties": dict(n=9, G=2, moves=4, open_plies=151, openings="mcts_tie_openings_9.json",
                            opts=dict(num_rollouts=119, num_rollouts_per_batch=14, virtual_loss=3, persistent_tree=1, c_puct=0.3,
                                      root_unexplored_q_zero=1, ply_pass_enabled=60, remove_pass_if_dangerous=1, komi=5.5)),
    # a positional-superko repetition two plies below the root: the recapture that closes the cycle makes a
    # terminal node inside the tree (GoState::terminated -> _check_superko, go_state.cc:96-111); the matching
    # record sits at an index that lanes beyond the board's 9 rows scan (superko_scan_warp)
    "9_superko_in_tree": dict(n=9, G=1, moves=3, open_plies=64, openings="mcts_superko_opening_9.json",
                              opts=dict(num_rollouts=96, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1, c_puct=5.0,
                                        komi=5.5, ply_pass_enabled=30)),
    # a net whose probabilities sit on a grid of 1/quant (bit-equal values among the legal moves of almost
    # every reply, as a half-precision network answers): the reference's pi2response leaves equal values in
    # the order of libstdc++'s std::sort, which the searches reproduce with std_sort_ties (the compiled
    # reference always sorts that way and takes no such option)
    "9_equal_priors": dict(n=9, G=3, moves=5, open_plies=20, quant=64, std_sort_ties=1,
                           opts=dict(num_rollouts=96, num_rollouts_per_batch=6, virtual_loss=1, persistent_tree=1, c_puct=1.5,
                                     ply_pass_enabled=40)),
    "19_equal_priors": dict(n=19, G=1, moves=3, open_plies=40, quant=256, std_sort_ties=1,
                            opts=dict(num_rollouts=128, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1, c_puct=1.5)),
}


def quantised_fakenet(n, quant):
    """the fake net with its probabilities on a grid of 1/quant: bit-equal values everywhere, as a
    half-precision network produces them"""
    def net(feats, hashes):
        pi, v = oracles.fakenet(hashes, n * n + 1)
        return (np.floor(pi * np.float32(quant)) / np.float32(quant)).astype(np.float32), v

    return net


def scenario_net(sc):
    """the scenario's network as a (feats, hashes) -> (pi, v) callback; None = the built-in fake net"""
    return quantised_fakenet(sc["n"], sc["quant"]) if "quant" in sc else None


def search_options(sc):
    """keyword arguments beyond sc["opts"] of the restatement, emulated and device searches of a scenario
    (the compiled reference always sorts like std::sort and takes no std_sort_ties)"""
    return {"std_sort_ties": sc["std_sort_ties"]} if "std_sort_ties" in sc else {}


def ref_mcts(sc):
    """the compiled reference search of a scenario"""
    return oracles.RefMcts(sc["n"], callback=scenario_net(sc), **sc["opts"])


def oracle_mcts(sc, lib=None):
    """the C restatement of the search for a scenario"""
    return oracles.OracleMcts(sc["n"], lib=lib, callback=scenario_net(sc), **search_options(sc), **sc["opts"])


def duplicate_prior_share(results):
    """share of root tables (run_search results) in which two root edges have bit-equal priors"""
    dup = 0
    for r in results:
        p = r["prior"][r["visits"] >= 0]
        dup += len(np.unique(p)) < len(p)
    return dup / len(results)


def scenario_openings(sc):
    """explicit opening move lists of a scenario ([G][open_plies] actions) or None (random openings)"""
    if "openings" not in sc:
        return None
    return json.load(open(os.path.join(GOLD, sc["openings"])))["openings"]


def opening(n, G, open_plies, make, fixed=None):
    rng = np.random.default_rng(5 + n)
    states = [make() for _ in range(G)]
    for t in range(open_plies):
        for g, s in enumerate(states):
            if fixed is not None:
                assert s.forward(int(fixed[g][t]))
                continue
            idx = np.flatnonzero(s.legal())
            assert s.forward(int(rng.choice(idx)))
    return states


def run_search(sc, make_state, make_mcts, forced=None, orders=None):
    """search `moves` moves in each of G games; the move played is the searcher's own choice or,
    when `forced` (a list in the same order as the returned results) is given, that action -- used to
    keep two implementations on the same trajectory when they break a most-visited TIE differently
    (the reference resolves ties by unordered_map order, tree_search_base.h:237-294)"""
    states = opening(sc["n"], sc["G"], sc["open_plies"], make_state, scenario_openings(sc))
    ms = [make_mcts() for _ in range(sc["G"])]
    out = []
    for _ in range(sc["moves"]):
        for s, m in zip(states, ms):
            r = m.act(s)
            a = r["best_action"] if forced is None else forced[len(out)]
            if orders is not None:
                orders.append(m.last_order())
            out.append(r)
            s.forward(a)
    return out, sum(m.num_evals() for m in ms)


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_restatement_equals_reference(name, oracle_lib):
    sc = SCENARIOS[name]
    n = sc["n"]
    if not oracles.have_ref(n):
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    oa, ob = [], []
    a, ea = run_search(sc, lambda: oracles.Ref(n), lambda: ref_mcts(sc), orders=oa)
    b, eb = run_search(sc, lambda: oracles.Oracle(n, oracle_lib), lambda: oracle_mcts(sc, oracle_lib),
                       forced=[r["best_action"] for r in a], orders=ob)
    assert ea == eb
    if "quant" in sc:  # the scenario reaches the equal-prior tie-breaks at the root
        assert duplicate_prior_share(a) >= 0.9, duplicate_prior_share(a)
    for i, (ra, rb) in enumerate(zip(a, b)):
        # the most-visited move is the first maximum in the reference's container order: same move, ties included
        assert ra["best_action"] == rb["best_action"], i
        np.testing.assert_array_equal(oa[i], ob[i], err_msg=f"container order, step {i}")
        np.testing.assert_array_equal(ra["visits"], rb["visits"], err_msg=f"step {i}")
        np.testing.assert_array_equal(ra["prior"], rb["prior"], err_msg=f"step {i}")
        np.testing.assert_allclose(ra["wsum"], rb["wsum"], rtol=0, atol=1e-4)
        assert ra["total_visits"] == rb["total_visits"]
        assert ra["root_value"] == rb["root_value"]


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_restatement_equals_golden(name, oracle_lib):
    path = os.path.join(GOLD, f"mcts_{name}.json")
    gold = json.load(open(path))
    sc = SCENARIOS[name]
    n = sc["n"]
    b, eb = run_search(sc, lambda: oracles.Oracle(n, oracle_lib), lambda: oracle_mcts(sc, oracle_lib),
                       forced=[st["best_action"] for st in gold["steps"]])
    assert eb == gold["num_evals"]
    assert len(b) == len(gold["steps"])
    for r, gsv in zip(b, gold["steps"]):
        assert r["best_action"] == gsv["best_action"]  # ties included (container order)
        assert r["total_visits"] == gsv["total_visits"]
        vis = {int(a): int(v) for a, v in zip(np.flatnonzero(r["visits"] >= 0), r["visits"][r["visits"] >= 0])}
        assert vis == {int(k): v for k, v in gsv["visits"].items()}


def test_restatement_equals_reference_on_random_option_sets(oracle_lib):
    """fuzz over the search options (rollouts, batch, virtual loss, c_puct, FPU switches, pass
    rules, tree persistence) and opening lengths: the C restatement must reproduce the reference
    search's root tables exactly in every configuration."""
    if not oracles.have_ref(9):
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    rng = np.random.default_rng(2026)
    for case in range(14):
        opts = dict(
            num_rollouts=int(rng.integers(8, 90)), num_rollouts_per_batch=int(rng.integers(1, 9)),
            virtual_loss=int(rng.integers(0, 4)), persistent_tree=int(rng.integers(0, 2)),
            c_puct=float(rng.choice([0.5, 0.85, 1.5, 2.5, 5.0])), unexplored_q_zero=int(rng.integers(0, 2)),
            root_unexplored_q_zero=int(rng.integers(0, 2)), ply_pass_enabled=int(rng.choice([0, 30, 70])),
            remove_pass_if_dangerous=int(rng.integers(0, 2)), komi=float(rng.choice([5.5, 6.5, 7.5])))
        sc = dict(n=9, G=2, moves=4, open_plies=int(rng.integers(0, 75)), opts=opts)
        a, ea = run_search(sc, lambda: oracles.Ref(9), lambda: oracles.RefMcts(9, **opts))
        b, eb = run_search(sc, lambda: oracles.Oracle(9, oracle_lib), lambda: oracles.OracleMcts(9, lib=oracle_lib, **opts),
                           forced=[r["best_action"] for r in a])
        assert ea == eb, (case, opts)
        for i, (ra, rb) in enumerate(zip(a, b)):
            assert ra["best_action"] == rb["best_action"], (case, i, opts)
            np.testing.assert_array_equal(ra["visits"], rb["visits"], err_msg=f"case {case} step {i} {opts}")
            np.testing.assert_array_equal(ra["prior"], rb["prior"], err_msg=f"case {case} step {i}")
            assert ra["root_value"] == rb["root_value"]


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_selected_prefix_property(name, oracle_lib):
    """k_select scans only edges [0, n_touched] of the prior-sorted list.  The restatement scans all
    edges (as the reference does) and counts every descent step whose full arg-max is not inside
    that prefix, or that finds a selected edge outside it: must never happen."""
    sc = SCENARIOS[name]
    n = sc["n"]
    states = opening(n, sc["G"], sc["open_plies"], lambda: oracles.Oracle(n, oracle_lib), scenario_openings(sc))
    ms = [oracle_mcts(sc, oracle_lib) for _ in range(sc["G"])]
    for _ in range(sc["moves"]):
        for s, m in zip(states, ms):
            s.forward(m.act(s)["best_action"])
    viol = sum(m.prefix_stats()[0] for m in ms)
    checks = sum(m.prefix_stats()[1] for m in ms)
    assert checks > 500 and viol == 0, (viol, checks)
    if name.endswith("_ties"):  # these scenarios are there for the container-order tie-break
        ties, beyond = sum(m.tie_stats()[0] for m in ms), sum(m.tie_stats()[1] for m in ms)
        assert ties > 0 and (beyond > 0 or name == "9_rounding_ties"), (ties, beyond)


@pytest.mark.parametrize("quant", [16, 256, 4096])
def test_equal_priors_in_std_sort_order(quant, oracle_lib):
    """std_sort_ties: moves with bit-equal probabilities are stored in the order libstdc++'s std::sort
    leaves them in pi2response (go/mcts/mcts.h:289-295) -- with it the restatement reproduces the compiled
    reference's visit tables on networks whose replies are full of equal values"""
    n = 9
    if not oracles.have_ref(n):
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    rng = np.random.default_rng(quant)
    for case in range(4):
        opts = dict(num_rollouts=int(rng.integers(20, 100)), num_rollouts_per_batch=int(rng.integers(1, 9)),
                    virtual_loss=int(rng.integers(0, 3)), persistent_tree=1, c_puct=float(rng.choice([0.5, 1.5])),
                    ply_pass_enabled=int(rng.choice([0, 40])))
        ref, o = oracles.Ref(n), oracles.Oracle(n, oracle_lib)
        rm = oracles.RefMcts(n, callback=quantised_fakenet(n, quant), **opts)
        om = oracles.OracleMcts(n, lib=oracle_lib, callback=quantised_fakenet(n, quant), std_sort_ties=1, **opts)
        for _ in range(int(rng.integers(0, 60))):
            a = int(rng.choice(np.flatnonzero(ref.legal())))
            assert ref.forward(a) and o.forward(a)
        for mv in range(4):
            w, p = rm.act(ref), om.act(o)
            np.testing.assert_array_equal(w["visits"], p["visits"], err_msg=f"quant {quant} case {case} move {mv}")
            np.testing.assert_array_equal(w["prior"], p["prior"])
            np.testing.assert_array_equal(rm.last_order(), om.last_order())
            assert w["best_action"] == p["best_action"]
            assert ref.forward(w["best_action"]) and o.forward(w["best_action"])
