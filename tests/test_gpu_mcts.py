"""GPU parity of the batched tree search (CUDA, through the C ABI) against the oracle: the C
restatement (oracle/mcts_oracle.c, itself pinned exactly to the compiled reference search) and the
UNMODIFIED reference search itself (oracle/_ref when built, else its root tables stored in tests/golden).  One search thread, fixed
rollouts per batch, rotation_flip off, deterministic fake net (oracle/fakenet.h).
Bar: root visit counts equal edge for edge (deviation 0), priors bit-identical, edge reward sums within
the last bits that the edge storage order can move (DESIGN.md, "Search semantics", deviation (i))."""
import json
import os

import numpy as np
import pytest

from tests import oracles
from tests.test_mcts_oracle_vs_ref import (GOLD, SCENARIOS, oracle_mcts, ref_mcts, scenario_net, scenario_openings,
                                           search_options)

pytestmark = pytest.mark.gpu


def fake_actor(mcts, n, net=None):
    """the network callback of a search: `net(feats, hashes)` (default: the hash-keyed fake net) on the
    hashes of the claimed leaves"""
    import torch

    def actor(batch):
        h, _, _ = mcts.leaf_info()
        pi, v = oracles.fakenet(h, n * n + 1) if net is None else net(None, h)
        assert batch["s"].shape[0] == len(h)
        return {"pi": torch.from_numpy(pi).to(mcts.device), "V": torch.from_numpy(v).to(mcts.device)}

    return actor


class GoldenMcts:
    """the compiled reference search's root tables of one game, replayed from tests/golden/mcts_<name>.json
    (scripts/gen_golden.py: steps in [move][game] order, games played on the reference's own choice)"""

    def __init__(self, steps, g, G, n, evals):
        self.steps, self.P1, self.evals = steps[g::G], n * n + 1, evals
        self.k = 0

    def act(self, state):
        st = self.steps[self.k]
        self.k += 1
        v = np.full(self.P1, -1, np.int64)
        for a, c in st["visits"].items():
            v[int(a)] = c
        return {"visits": v, "total_visits": st["total_visits"], "best_action": st["best_action"]}

    def num_evals(self):
        return self.evals


def root_wsum(mc):
    """float32 [G, N*N+1]: reward sum of every root edge by action (0 where there is no edge)"""
    e = mc.root_edges()
    w = np.zeros_like(e["wsum"])
    for g in range(len(w)):
        k = e["n_edges"][g]
        w[g, e["actions"][g, :k].astype(np.int64)] = e["wsum"][g, :k]
    return w


def run_gpu_vs_cpu(sc, use_ref, golden=None, std_sort_ties=None, compare=True):
    """the device search against the compiled reference (use_ref), the C restatement or the reference's
    stored root tables (golden), move after move on the reference's own choice.  The bar is exact: equal
    root visit tables, totals, values and moves; priors bit-identical and edge reward sums within the
    last-bit deviation of the storage order (DESIGN.md, deviation (i)) when a live search is the
    comparison.  compare=False: assert nothing about the tables, return how many differ."""
    import elf_b200

    n, G = sc["n"], sc["G"]
    rng = np.random.default_rng(5 + n)
    gb = elf_b200.GoBatch(G, board_size=n)
    make = (lambda: oracles.Ref(n)) if use_ref else (lambda: oracles.Oracle(n))
    states = [make() for _ in range(G)]
    fixed = scenario_openings(sc)  # explicit opening move lists (the tie scenarios) or None
    for t in range(sc["open_plies"]):
        acts = np.empty(G, np.int32)
        for g, s in enumerate(states):
            idx = np.flatnonzero(s.legal())
            acts[g] = int(fixed[g][t]) if fixed is not None else int(rng.choice(idx))
            assert s.forward(acts[g])
        assert gb.forward(acts).all()
    sst = search_options(sc) if std_sort_ties is None else {"std_sort_ties": std_sort_ties}
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, **sst, **sc["opts"])
    if golden is not None:
        cpu = [GoldenMcts(golden["steps"], g, G, n, golden["num_evals"] if g == 0 else 0) for g in range(G)]
    else:
        cpu = [ref_mcts(sc) if use_ref else oracle_mcts(sc) for _ in range(G)]
    actor = fake_actor(mc, n, scenario_net(sc))
    tables, differ = 0, 0
    for mv in range(sc["moves"]):
        res = mc.act(actor)
        pri, wsum = mc.root_priors(), root_wsum(mc)
        acts = np.empty(G, np.int32)
        for g in range(G):
            rr = cpu[g].act(states[g])
            gv, rv = res["visits"][g], rr["visits"]
            tables += 1
            if not compare:
                differ += not (np.array_equal(gv, rv) and (golden is not None or np.array_equal(pri[g], np.where(
                    rv >= 0, rr["prior"], np.float32(-1)))))
            else:
                assert ((gv >= 0) == (rv >= 0)).all(), f"edge sets differ: move {mv} game {g}"
                np.testing.assert_array_equal(gv, rv, err_msg=f"root visits, move {mv} game {g}")
                assert res["total_visits"][g] == rr["total_visits"]
                # an exact most-visited tie resolves in the reference's container order, on the device too
                assert res["best_action"][g] == rr["best_action"], f"move {mv} game {g}"
                if golden is None:  # the stored tables hold visits, totals and the chosen move only
                    has = rv >= 0
                    assert res["root_value"][g] == np.float32(rr["root_value"])
                    assert abs(res["best_q"][g] - rr["best_q"]) < 1e-5
                    np.testing.assert_array_equal(pri[g][has], rr["prior"][has], err_msg=f"priors, move {mv} game {g}")
                    np.testing.assert_allclose(wsum[g][has], rr["wsum"][has], rtol=0, atol=1e-4,
                                               err_msg=f"edge reward sums, move {mv} game {g}")
            acts[g] = rr["best_action"]
            assert states[g].forward(acts[g])
        assert gb.forward(acts).all()
        mc.advance(acts)
    assert (mc.errors() == 0).all(), mc.errors()
    if compare:
        assert mc.eval_count() == sum(c.num_evals() for c in cpu)
    mc.close()
    gb.close()
    return tables, differ


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_gpu_search_vs_restatement(name):
    tables, _ = run_gpu_vs_cpu(SCENARIOS[name], use_ref=False)
    print(f"{name}: {tables} root tables equal")


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_gpu_search_vs_reference(name):
    """against the compiled reference search when oracle/_ref is built, else against its stored root tables"""
    if oracles.have_ref(SCENARIOS[name]["n"]):
        run_gpu_vs_cpu(SCENARIOS[name], use_ref=True)
    else:
        golden = json.load(open(os.path.join(GOLD, f"mcts_{name}.json")))
        run_gpu_vs_cpu(SCENARIOS[name], use_ref=False, golden=golden)


def test_equal_priors_scenario_needs_std_sort_ties():
    """negative control of the *_equal_priors scenarios: without std_sort_ties (equal probabilities stored
    by ascending move, not in std::sort's order) the device search must leave the reference's root tables
    somewhere -- the scenario does reach the equal-prior tie-breaks"""
    sc = SCENARIOS["9_equal_priors"]
    if oracles.have_ref(sc["n"]):
        tables, differ = run_gpu_vs_cpu(sc, use_ref=True, std_sort_ties=0, compare=False)
    else:
        golden = json.load(open(os.path.join(GOLD, "mcts_9_equal_priors.json")))
        tables, differ = run_gpu_vs_cpu(sc, use_ref=False, golden=golden, std_sort_ties=0, compare=False)
    print(f"std_sort_ties=0: {differ} of {tables} root tables differ from the reference")
    assert differ >= 1


def test_gpu_search_many_games_batched():
    """64 games searched together must give each game exactly what it gets alone (games are
    independent; the leaf batch interleaves them)."""
    import elf_b200

    n, G = 9, 64
    opts = dict(num_rollouts=64, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1, c_puct=1.5)
    gb = elf_b200.GoBatch(G, board_size=n)
    os_ = [oracles.Oracle(n) for _ in range(G)]
    rng = np.random.default_rng(11)
    for _ in range(20):
        acts = np.empty(G, np.int32)
        for g, s in enumerate(os_):
            idx = np.flatnonzero(s.legal())
            acts[g] = int(rng.choice(idx))
            s.forward(acts[g])
        gb.forward(acts)
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, **opts)
    cpu = [oracles.OracleMcts(n, **opts) for _ in range(G)]
    for mv in range(3):
        res = mc.act(fake_actor(mc, n))
        acts = np.empty(G, np.int32)
        for g in range(G):
            rr = cpu[g].act(os_[g])
            np.testing.assert_array_equal(res["visits"][g], rr["visits"], err_msg=f"move {mv} game {g}")
            assert res["best_action"][g] == rr["best_action"] and res["total_visits"][g] == rr["total_visits"]
            acts[g] = rr["best_action"]
            os_[g].forward(acts[g])
        gb.forward(acts)
        mc.advance(acts)
    assert (mc.errors() == 0).all()


def test_gpu_search_inactive_and_reset():
    import elf_b200

    n, G = 9, 4
    gb = elf_b200.GoBatch(G, board_size=n)
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, num_rollouts=32, num_rollouts_per_batch=4)
    res = mc.act(fake_actor(mc, n), active=np.array([1, 0, 1, 0], np.uint8))
    assert res["best_action"][1] == -1 and res["best_action"][3] == -1
    assert res["total_visits"][0] == 28 and res["total_visits"][2] == 28  # first wave expands the root
    mc.reset(np.array([1, 0, 0, 0], np.uint8))
    res2 = mc.act(fake_actor(mc, n))
    assert res2["total_visits"][0] == 28            # tree dropped: root expanded again
    assert res2["total_visits"][2] == 28 + 32       # tree kept (same root: no move was played)
    assert res2["total_visits"][1] == 28


def test_rotation_flip_is_a_pure_relabelling():
    """rotation_flip draws a D4 code per evaluation: the features are written under that symmetry
    and the policy is mapped back through the inverse (board_feature.h:97-144).  A net that answers
    in BOARD coordinates, pushed through the forward symmetry by the test, must therefore give
    exactly the search it gives without rotation."""
    import torch
    import elf_b200

    n, G = 9, 6
    P = n * n
    opts = dict(num_rollouts=96, num_rollouts_per_batch=4, virtual_loss=1, persistent_tree=1, c_puct=1.5)

    def fwd(d4, x, y):  # BoardFeature::Transform
        rot, flip = d4 & 3, d4 >> 2
        if rot == 1:
            a, b = y, n - x - 1
        elif rot == 2:
            a, b = n - x - 1, n - y - 1
        elif rot == 3:
            a, b = n - y - 1, x
        else:
            a, b = x, y
        return (b, a) if flip else (a, b)

    perm = np.zeros((8, P + 1), np.int64)  # perm[d4][nn_action] = board_action
    for d4 in range(8):
        for x in range(n):
            for y in range(n):
                tx, ty = fwd(d4, x, y)
                perm[d4][tx * n + ty] = x * n + y
        perm[d4][P] = P

    def run(rotation):
        gb = elf_b200.GoBatch(G, board_size=n)
        rng = np.random.default_rng(3)
        os_ = [oracles.Oracle(n) for _ in range(G)]
        for _ in range(16):
            acts = np.empty(G, np.int32)
            for g, s in enumerate(os_):
                idx = np.flatnonzero(s.legal())
                acts[g] = int(rng.choice(idx))
                s.forward(acts[g])
            gb.forward(acts)
        mc = elf_b200.MctsBatch(gb, rotation_flip=rotation, seed=5, **opts)
        feats_seen = []

        def actor(batch):
            h, _, _ = mc.leaf_info()
            pi_board, v = oracles.fakenet(h, P + 1)
            d4 = mc.leaf_d4
            if rotation:
                assert len(set(d4.tolist())) > 1
            pi_nn = np.take_along_axis(pi_board, perm[d4], axis=1)  # pi_nn[a] = pi_board[board(a)]
            feats_seen.append(batch["s"].sum().item())
            return {"pi": torch.from_numpy(pi_nn).to(mc.device), "V": torch.from_numpy(v).to(mc.device)}

        out = []
        for _ in range(3):
            res = mc.act(actor)
            out.append(res["visits"].copy())
            a = res["best_action"]
            gb.forward(a)
            mc.advance(a)
        return out, feats_seen

    a, fa = run(0)
    b, fb = run(1)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert fa == fb  # plane sums are invariant under the symmetry


def test_selfplay_driver_smoke():
    """GoGameSelfPlay::act mirror: a few moves of real self-play with a small random-init net:
    legal moves only, games restart on termination, counters consistent."""
    import torch
    import elf_b200
    from elf_b200.model import Actor, PolicyValueNet

    torch.manual_seed(0)
    n, G = 9, 32
    net = PolicyValueNet(n, num_block=2, dim=32).cuda()
    sp = elf_b200.selfplay.SelfPlay(Actor(net, batchsize=64, dtype=torch.float32, channels_last=False), num_games=G, board_size=n, policy_distri_cutoff=4,
                                    num_rollouts=32, num_rollouts_per_batch=4, move_cutoff=30, seed=1,
                                    record_games=True)
    total = 0
    for _ in range(36):
        total += sp.step()
    assert total == sp.moves_played and total > 30 * G
    assert sp.games_finished >= G  # move_cutoff 30 forces restarts
    assert all(abs(fv) <= n * n + 7.5 for fv, _, _ in sp.results)
    assert (sp.mcts.errors() == 0).all()
    # reference-format records: one per finished game, policies for the first `cutoff` plies only
    assert len(sp.records) == sp.games_finished
    # (a game may end early by two passes: among equally visited moves the reference's container order
    # puts pass, key 0, first -- most games run into move_cutoff)
    assert sum(r["result"]["num_move"] >= 28 for r in sp.records) >= G // 2
    r0 = max(sp.records, key=lambda r: r["result"]["num_move"])["result"]
    assert r0["content"].startswith("(;B[") and len(r0["policies"]) == 4 and len(r0["policies"][0]) == 121
    assert len(r0["values"]) >= r0["num_move"] >= 28
    sp.close()


@pytest.mark.parametrize("n,open_plies", [(9, 30), (19, 12)])
def test_leaf_features_match_reference_extractor(n, open_plies):
    """The planes handed to the network for every MCTS leaf (history gathered along the tree's
    parent chain + the game's ring) must equal what the reference's BoardFeature::extractAGZ
    produces for the same leaf state.  The reference search runs with a recording callback; every
    GPU leaf must reproduce one of the reference's recorded (hash -> planes) entries exactly."""
    import torch
    import elf_b200

    if not oracles.have_ref(n):
        pytest.skip("oracle/_ref not built")
    G = 3
    P1 = n * n + 1
    opts = dict(num_rollouts=64, num_rollouts_per_batch=4, virtual_loss=1, persistent_tree=1, c_puct=1.5)
    rng = np.random.default_rng(21)
    gb = elf_b200.GoBatch(G, board_size=n)
    refs = [oracles.Ref(n) for _ in range(G)]
    for _ in range(open_plies):
        acts = np.empty(G, np.int32)
        for g, r in enumerate(refs):
            idx = np.flatnonzero(r.legal())
            acts[g] = int(rng.choice(idx))
            r.forward(acts[g])
        gb.forward(acts)
    recorded = {}

    def ref_cb(feats, hashes):
        for f, h in zip(feats, hashes):
            recorded.setdefault(int(h), []).append(f.copy())
        return oracles.fakenet(hashes, P1)

    rms = [oracles.RefMcts(n, callback=ref_cb, **opts) for _ in range(G)]
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, **opts)
    checked = [0]

    def actor(batch):
        h, _, _ = mc.leaf_info()
        s = batch["s"].cpu().numpy()
        for i, hh in enumerate(h):
            cands = recorded.get(int(hh))
            assert cands, "GPU evaluated a state the reference never evaluated"
            assert any((s[i] == c).all() for c in cands), f"feature planes differ for leaf hash {int(hh):x}"
            checked[0] += 1
        pi, v = oracles.fakenet(h, P1)
        return {"pi": torch.from_numpy(pi).to(mc.device), "V": torch.from_numpy(v).to(mc.device)}

    for mv in range(4):
        ref_res = [rms[g].act(refs[g]) for g in range(G)]  # reference first: fills `recorded`
        res = mc.act(actor)
        acts = np.array([r["best_action"] for r in ref_res], np.int32)
        for g in range(G):
            assert np.abs(res["visits"][g] - ref_res[g]["visits"]).max() == 0
            refs[g].forward(acts[g])
        gb.forward(acts)
        mc.advance(acts)
    assert checked[0] > 300


@pytest.mark.parametrize("alpha", [0.03, 2.0])
def test_root_dirichlet_noise(alpha):
    """NodeT::enhanceExploration: P <- (1-eps) P + eps * Dir(alpha) on a root that already has
    edges; nothing on a fresh (unexpanded) root.  Streams differ from the reference's mt19937, so
    the check is distributional: the mixed-in vector is non-negative, sums to 1, has the Dirichlet
    mean 1/n and variance (n-1)/(n^2 (n alpha + 1)); and the search still accounts for every rollout."""
    import elf_b200

    n, G, eps = 9, 96, 0.25
    gb = elf_b200.GoBatch(G, board_size=n)
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, num_rollouts=32, num_rollouts_per_batch=4, root_epsilon=eps,
                            root_alpha=alpha, seed=11)
    actor = fake_actor(mc, n)
    res = mc.act(actor)  # move 1: the root is unexpanded when the search starts -> no noise
    a = res["best_action"]
    assert res["total_visits"].tolist() == [28] * G
    gb.forward(a)
    mc.advance(a)
    before = mc.root_priors()          # the kept child: expanded, priors straight from pi2response
    mc.begin_move()                    # noise goes in here
    after = mc.root_priors()
    has = before >= 0
    assert (has == (after >= 0)).all() and has.sum(1).min() >= 60
    d = np.where(has, (after - (1 - eps) * before) / eps, 0.0).astype(np.float64)
    assert (d > -1e-6).all()
    np.testing.assert_allclose(d.sum(1), 1.0, atol=1e-4)
    k = has.sum(1)
    mean = (d.sum(1) / k)
    np.testing.assert_allclose(mean, 1.0 / k, rtol=1e-3)
    var_emp = np.mean([(d[g][has[g]] - 1.0 / k[g]).var() for g in range(G)])
    kk = k.mean()
    var_th = (kk - 1) / (kk * kk * (kk * alpha + 1))
    assert 0.6 * var_th < var_emp < 1.5 * var_th, (var_emp, var_th)
    # two games never get the same noise
    assert len({tuple(np.round(d[g][has[g]], 7)) for g in range(G)}) == G
    # finish the move through the flagged (full-scan) root
    for _ in range(mc.waves_per_move):
        s = mc.select()
        if s.shape[0]:
            gb.synchronize()
            r = actor({"s": s})
            mc.expand_backup(r["pi"], r["V"])
        else:
            mc.expand_backup(None, None)
    res2 = mc.results()
    assert (res2["total_visits"] >= 32).all()
    assert (mc.errors() == 0).all()


def test_gpu_search_with_a_real_network_matches_reference():
    """Full loop with a real (small, random-init, fp32) policy/value network: the reference search
    evaluates the net on the planes ITS extractor produced, the GPU search on the planes OUR leaf
    feature kernel produced; the same CPU network instance, one position per call (so results do not
    depend on batch composition).  Identical planes -> identical pi/V -> identical root visits."""
    import torch
    import elf_b200
    from elf_b200.model import PolicyValueNet

    n = 9
    if not oracles.have_ref(n):
        pytest.skip("oracle/_ref not built")
    torch.manual_seed(7)
    torch.set_num_threads(1)
    net = PolicyValueNet(n, num_block=2, dim=16).eval()
    G, P1 = 3, n * n + 1
    opts = dict(num_rollouts=96, num_rollouts_per_batch=4, virtual_loss=1, persistent_tree=1, c_puct=1.5)

    def eval_cpu(planes):  # planes: numpy [k,18,n,n]
        pis, vs = [], []
        with torch.no_grad():
            for i in range(planes.shape[0]):
                out = net(torch.from_numpy(np.ascontiguousarray(planes[i:i + 1])))
                pis.append(out["pi"][0].numpy().copy())
                vs.append(float(out["V"].reshape(-1)[0]))
        return np.stack(pis).astype(np.float32), np.array(vs, np.float32)

    rng = np.random.default_rng(31)
    gb = elf_b200.GoBatch(G, board_size=n)
    refs = [oracles.Ref(n) for _ in range(G)]
    for _ in range(24):
        acts = np.empty(G, np.int32)
        for g, r in enumerate(refs):
            idx = np.flatnonzero(r.legal())
            acts[g] = int(rng.choice(idx))
            r.forward(acts[g])
        gb.forward(acts)
    rms = [oracles.RefMcts(n, callback=lambda f, h: eval_cpu(f), **opts) for _ in range(G)]
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, **opts)

    def actor(batch):
        pi, v = eval_cpu(batch["s"].cpu().numpy())
        return {"pi": torch.from_numpy(pi).to(mc.device), "V": torch.from_numpy(v).to(mc.device)}

    for mv in range(4):
        res = mc.act(actor)
        pri = mc.root_priors()
        acts = np.empty(G, np.int32)
        for g in range(G):
            rr = rms[g].act(refs[g])
            np.testing.assert_array_equal(res["visits"][g], rr["visits"], err_msg=f"move {mv} game {g}")
            has = rr["visits"] >= 0
            np.testing.assert_array_equal(pri[g][has], rr["prior"][has], err_msg=f"priors, move {mv} game {g}")
            assert res["best_action"][g] == rr["best_action"]
            acts[g] = rr["best_action"]
            refs[g].forward(acts[g])
        gb.forward(acts)
        mc.advance(acts)


def test_node_pool_exhaustion_prunes_the_tree_and_keeps_searching():
    """bounded node pool (documented deviation): when a game's pool cannot hold one more move's
    worth of nodes, the subtrees under the root's least-visited children are recycled (counter in
    errors()[3]); the root keeps its edge statistics, the search carries on, rollouts are all
    accounted for, the pool never overflows during a descent (errors()[1] stays 0)."""
    import elf_b200

    n, G = 9, 6
    gb = elf_b200.GoBatch(G, board_size=n)
    R, B = 32, 4
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, num_rollouts=R, num_rollouts_per_batch=B, nodes_per_game=R + 8)
    actor = fake_actor(mc, n)
    prunes = 0
    for mv in range(8):
        res = mc.act(actor)
        tv = res["total_visits"]
        assert ((tv == R - B) | (tv >= R)).all()  # fresh root (first wave expands it) or reused tree
        a = res["best_action"]
        assert gb.forward(a).all()
        mc.advance(a)
        e = mc.errors()
        assert e[0] == 0 and e[1] == 0 and e[2] == 0, e
        prunes = int(e[3])
    assert prunes > 0  # the small pool must have forced at least one pruning
    mc.close()
    gb.close()


def test_root_mismatch_raises_like_the_reference():
    """TreeSearchT::setRootNodeState throws when the persistent root is not the position it is asked
    to search (tree_search.h:488-492).  Here: the board moves without advance() -> begin_move raises,
    the stale tree is gone and the next search starts from the board."""
    import elf_b200
    from elf_b200.lib import ElfB200Error

    n, G = 9, 3
    gb = elf_b200.GoBatch(G, board_size=n)
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, num_rollouts=16, num_rollouts_per_batch=4)
    actor = fake_actor(mc, n)
    res = mc.act(actor)
    assert gb.forward(res["best_action"]).all()  # no mc.advance(): the trees are stale now
    with pytest.raises(ElfB200Error, match="Root state is not the same"):
        mc.act(actor)
    res = mc.act(actor)  # rebuilt from the board
    assert (res["total_visits"] == 16 - 4).all() and mc.errors()[0] == G
    mc.close()
    gb.close()


@pytest.mark.parametrize("n", [9, 19])
def test_fast_feature_formats_async_waves_and_pipeline(n):
    """the same search four ways -- float32 features with a host wait per wave (baseline), binary16
    NHWC leaf features, waves without any host read-back (device-side leaf count), and two half
    batches interleaved by WavePipeline -- gives identical root statistics; the NHWC leaf batch equals
    the float32 one position by position."""
    import torch

    import elf_b200
    from elf_b200.pipeline import WavePipeline

    G, R, B = 8, 24, 4
    opts = dict(num_rollouts=R, num_rollouts_per_batch=B, rotation_flip=1, seed=3)

    def opening(gb, lo=0):
        rng = np.random.default_rng(1)
        os_ = [oracles.Oracle(n) for _ in range(G)]
        for _ in range(10):
            acts = np.array([int(rng.choice(np.flatnonzero(o.legal()))) for o in os_], np.int32)
            for o, a in zip(os_, acts):
                o.forward(int(a))
            gb.forward(acts[lo:lo + gb.num_games])

    def net(feat_f32, hashes):  # deterministic in the position, independent of the batch layout
        pi, v = oracles.fakenet(hashes, n * n + 1)
        return torch.from_numpy(pi), torch.from_numpy(v)

    def make(G_, lo=0, **kw):
        gb = elf_b200.GoBatch(G_, board_size=n)
        opening(gb, lo)
        return gb, elf_b200.MctsBatch(gb, **opts, **kw)

    def actor_for(mc, log=None):
        def actor(batch):
            h, gi, _ = mc.leaf_info()
            key = "s" if "s" in batch else "s_nhwc"
            if log is not None:
                x = batch[key][: len(h)]
                x = x.float().cpu().numpy() if key == "s" else x.float().permute(0, 3, 1, 2)[:, :18].cpu().numpy()
                # leaf slots are handed out by an atomic counter: their order is not reproducible between
                # runs on hardware, so a wave's batch is keyed by (game, position hash)
                log.append({(int(g_), int(h_)): x[i] for i, (g_, h_) in enumerate(zip(gi, h))})
            pi, v = net(None, h)
            full = batch[key].shape[0]
            P = torch.zeros(full, n * n + 1)
            V = torch.zeros(full)
            P[: len(h)], V[: len(h)] = pi, v
            return {"pi": P.to(mc.device), "V": V.to(mc.device)}
        return actor

    # note: the d4 code of an evaluation depends on (seed, game index, wave, node, hash): the halves of
    # the pipeline run are therefore compared with rotation-independent quantities (the fake net is
    # keyed by the hash and answers in NN action space, so visits differ with d4) -> rotation off there
    gb0, m0 = make(G)
    log0 = []
    r0 = m0.act(actor_for(m0, log0))
    gb1, m1 = make(G, feature_format="f16", cpad=24)
    log1 = []
    r1 = m1.act(actor_for(m1, log1))
    assert len(log0) == len(log1)
    for a, b in zip(log0, log1):
        assert a.keys() == b.keys()
        for k in a:
            np.testing.assert_array_equal(a[k], b[k])
    for k in ("visits", "best_action", "root_value", "total_visits"):
        np.testing.assert_array_equal(r0[k], r1[k])
    for m, g in ((m0, gb0), (m1, gb1)):
        assert (m.errors() == 0).all()
        m.close()
        g.close()
    # waves without any host read-back (fixed grids, device-side leaf count) with a net that reads the
    # planes, against the same net through the synchronous path
    def plane_actor(mc):
        def actor(batch):
            x = batch["s"] if "s" in batch else batch["s_nhwc"].float().permute(0, 3, 1, 2)[:, :18]
            pi, v = oracles.feature_net(x.float().cpu().numpy(), n * n + 1)
            return {"pi": torch.from_numpy(pi).to(mc.device), "V": torch.from_numpy(v).to(mc.device)}
        return actor

    gb2, m2 = make(G)
    r2 = m2.act(plane_actor(m2))
    gb3, m3 = make(G, feature_format="bf16", cpad=32)
    act3 = plane_actor(m3)
    m3.begin_move()
    for _ in range(m3.waves_per_move):
        s = m3.select(wait=False)
        assert s.shape[0] == m3.max_leaves
        m3.gb.synchronize()
        rep = act3({"s_nhwc": s})
        torch.cuda.synchronize()
        m3.expand_backup(rep["pi"], rep["V"])
    r3 = m3.results()
    for k in ("visits", "best_action", "root_value", "total_visits"):
        np.testing.assert_array_equal(r2[k], r3[k])
    assert m3.eval_count() == m2.eval_count()
    for m, g in ((m2, gb2), (m3, gb3)):
        assert (m.errors() == 0).all()
        m.close()
        g.close()
    # two halves through the pipeline == the two halves searched one after the other
    opts["rotation_flip"] = 0
    res_seq, res_pipe = [], []
    for mode in ("seq", "pipe"):
        parts = [make(G // 2, lo) for lo in (0, G // 2)]
        if mode == "seq":
            for gb, mc in parts:
                res_seq.append(mc.act(actor_for(mc)))
        else:
            class Routed:  # one callable for both parts, routed by the tensor it is handed
                batchsize = 0

                def __call__(self, batch):
                    for gb, mc in parts:
                        if batch["s"].data_ptr() == mc.feat.data_ptr():
                            return actor_for(mc)(batch)
                    raise AssertionError("unknown batch")
            pipe = WavePipeline([mc for _, mc in parts], Routed())
            pipe.search()
            res_pipe = [mc.results() for _, mc in parts]
        for gb, mc in parts:
            assert (mc.errors() == 0).all()
            mc.close()
            gb.close()
    for a, b in zip(res_seq, res_pipe):
        for k in ("visits", "best_action", "root_value", "total_visits"):
            np.testing.assert_array_equal(a[k], b[k])


def test_fused_actor_matches_module():
    """FusedActor on the GPU (cuDNN fused conv+bias(+add)+ReLU, CUDA graph for full batches, eager for
    the tail, float32 NCHW and binary16 NHWC inputs) against the float32 module"""
    import torch

    from elf_b200.model import FusedActor, PolicyValueNet
    from tests.test_fused_actor import randomise_bn

    torch.manual_seed(1)
    dev = torch.device("cuda")
    m = PolicyValueNet(9, num_block=3, dim=32).to(dev).eval()
    randomise_bn(m)
    fa = FusedActor(m, batchsize=8, dtype=torch.float16, cuda_graph=True)
    x = (torch.rand(21, 18, 9, 9, device=dev) > 0.6).float()
    with torch.no_grad():
        ref = m(x)
    for _ in range(2):  # replay twice: static buffers are reused
        out = fa({"s": x})
        assert (out["pi"] - ref["pi"]).abs().max().item() < 5e-3
        assert (out["V"] - ref["V"].reshape(-1)).abs().max().item() < 2e-2
    xn = torch.zeros(21, 9, 9, fa.cpad, dtype=torch.float16, device=dev)
    xn[..., :18] = x.permute(0, 2, 3, 1).half()
    out2 = fa({"s_nhwc": xn})
    assert torch.equal(out2["pi"], out["pi"]) and torch.equal(out2["V"], out["V"])


def test_device_move_choice_sampling_argmax_and_resign():
    """elfb200_mcts_choose: sample_multinomial over root visits while ply <= cutoff (empirical
    frequencies follow N/sum N), most visited afterwards, resignation rule of ResignCheck."""
    import elf_b200

    n, G = 9, 512
    gb = elf_b200.GoBatch(G, board_size=n)      # 512 identical games (empty board)
    mc = elf_b200.MctsBatch(gb, rotation_flip=0, num_rollouts=64, num_rollouts_per_batch=4)
    res = mc.act(fake_actor(mc, n))
    v = res["visits"][0]
    assert (res["visits"] == v).all()           # identical games -> identical root tables
    # beyond the cutoff: the most visited move, for every game
    a, val = mc.choose(policy_distri_cutoff=0, resign_thres=0.05, seed=1)
    assert (a == res["best_action"]).all()
    np.testing.assert_allclose(val, res["best_q"], rtol=0, atol=1e-6)
    # within the cutoff: sampled ~ visits (different games draw different moves)
    counts = np.zeros(n * n + 1)
    for seed in range(8):
        a, _ = mc.choose(policy_distri_cutoff=5, resign_thres=0.05, seed=seed)
        assert (v[a] > 0).all()                 # only visited edges can be drawn
        counts += np.bincount(a, minlength=n * n + 1)
    p = np.maximum(v, 0) / np.maximum(v, 0).sum()
    big = p > 0.03
    np.testing.assert_allclose(counts[big] / counts.sum(), p[big], rtol=0.25)
    assert len(np.unique(a)) > 3
    # resign: needs ply >= 50 and value below -1 + thres; with thres = 2 every value qualifies
    a, _ = mc.choose(policy_distri_cutoff=0, resign_thres=2.0, seed=1)
    assert (a == res["best_action"]).all()      # ply 1 < 50: nobody resigns
    gb2 = elf_b200.GoBatch(4, board_size=n)
    os_ = [oracles.Oracle(n) for _ in range(4)]
    rng = np.random.default_rng(0)
    for _ in range(52):
        acts = np.empty(4, np.int32)
        for g, s in enumerate(os_):
            idx = np.flatnonzero(s.legal() & (1 - s.true_eyes(int(s.info()[1]))))
            acts[g] = int(rng.choice(idx)) if len(idx) else n * n
            s.forward(acts[g])
        gb2.forward(acts)
    mc2 = elf_b200.MctsBatch(gb2, rotation_flip=0, num_rollouts=32, num_rollouts_per_batch=4)
    mc2.act(fake_actor(mc2, n))
    a, _ = mc2.choose(policy_distri_cutoff=0, resign_thres=2.0, never_resign=np.array([0, 1, 0, 1], np.uint8), seed=1)
    assert a[0] == -1 and a[2] == -1 and a[1] >= 0 and a[3] >= 0
    a, _ = mc2.choose(policy_distri_cutoff=0, resign_thres=0.0, seed=1)
    assert (a >= 0).all()                        # value can never be below -1
    # the same decisions from the reference's own ResignCheck (game_utils.h:15-54) through
    # GoStateExt::shouldResign and the ply test of GoGameSelfPlay::act: 64 games around ply 50 with both
    # colours to move, a spread of predicted values, several thresholds, mixed never-resign flags
    if oracles.have_ref(n):
        G3 = 64
        gb3 = elf_b200.GoBatch(G3, board_size=n)
        os3 = [oracles.Oracle(n) for _ in range(G3)]
        for t in range(51):
            acts = np.full(G3, -1, np.int32)
            for g, s_ in enumerate(os3):
                if t >= 47 + g % 4:   # games stop at plies 48..51: both sides of the ply-50 test, both colours
                    continue
                idx = np.flatnonzero(s_.legal() & (1 - s_.true_eyes(int(s_.info()[1]))))
                acts[g] = int(rng.choice(idx)) if len(idx) else n * n
                s_.forward(acts[g])
            gb3.forward(acts)
        info = gb3.info()
        assert set(info[:, 1]) == {1, 2} and info[:, 0].min() < 50 <= info[:, 0].max()
        mc3 = elf_b200.MctsBatch(gb3, rotation_flip=0, num_rollouts=32, num_rollouts_per_batch=4)
        mc3.act(fake_actor(mc3, n))
        never = (np.arange(G3) % 3 == 0).astype(np.uint8)
        decided = 0
        for thres in (0.05, 0.4, 0.9, 1.3, 2.0):
            a, val = mc3.choose(policy_distri_cutoff=0, resign_thres=thres, never_resign=never, seed=1)
            for g in range(G3):
                want = oracles.ref_should_resign(thres, never[g], val[g], info[g, 1], info[g, 0], n)
                assert (a[g] == -1) == want, (thres, g, val[g], info[g, :2], never[g])
                decided += want
        assert decided > 20
        mc3.close()
        gb3.close()


def test_selfplay_soak_tree_reuse_over_many_moves():
    """long run of the full loop (search, device move choice, forward, tree advance, game end,
    restart) with the fake network: many games end and restart, the node pools never overflow or
    drop a tree, no root/hash inconsistency is ever detected."""
    import torch
    import elf_b200

    n, G = 9, 32
    sp = elf_b200.selfplay.SelfPlay(None, num_games=G, board_size=n, policy_distri_cutoff=6, resign_thres=0.05,
                                    never_resign_ratio=0.5, num_rollouts=32, num_rollouts_per_batch=4, seed=4,
                                    rotation_flip=1, record_games=True, move_cutoff=45)

    def actor(batch):
        h, _, _ = sp.mcts.leaf_info()
        pi, v = oracles.fakenet(h, n * n + 1)
        # the fake policy is expressed in NN coordinates here; under rotation_flip the engine maps it
        # back through the inverse D4 -- any permutation is a valid policy for a soak test
        return {"pi": torch.from_numpy(pi).to(sp.mcts.device), "V": torch.from_numpy(v).to(sp.mcts.device)}

    sp.actor = actor
    moves = 0
    for _ in range(100):
        moves += sp.step()
    assert sp.games_finished >= G            # every slot finished at least one game on average
    assert moves == sp.moves_played
    e = sp.mcts.errors()
    assert (e == 0).all(), e
    reasons = {r for _, _, r in sp.results}
    assert "two_pass" in reasons or "resign" in reasons or "max_step" in reasons
    assert len(sp.records) == sp.games_finished
    for rec in sp.records[:20]:
        assert rec["result"]["num_move"] == rec["result"]["content"].count(";")
    sp.close()


@pytest.mark.parametrize("n", [9, 19])
def test_gpu_selfplay_records_are_accepted_by_the_reference_parser(n):
    """row f1 on the device: records written by GPU self-play (real search, real visit tables) go
    through the compiled reference's own Record::createFromJson / setJsonFields (oracle/_ref,
    ref_offline_shim.cc; JSON_LOAD throws on any missing field) and come back field for field; the
    batch parser keeps all of them; the u8-quantised policies equal GoStateExt::addMCTSPolicy's on
    the same visit counts; and replaying a record's moves on reference boards reproduces the game."""
    import json

    import torch

    import elf_b200
    from elf_b200 import record
    from elf_b200.model import Actor, PolicyValueNet
    from tests.test_replay_records import same

    if not oracles.have_ref(n):
        pytest.skip("oracle/_ref not built")
    torch.manual_seed(2)
    G = 12 if n == 9 else 6
    net = PolicyValueNet(n, num_block=1, dim=16).cuda()
    cutoff = 6
    sp = elf_b200.selfplay.SelfPlay(Actor(net, batchsize=64, dtype=torch.float32, channels_last=False), num_games=G,
                                    board_size=n, policy_distri_cutoff=cutoff, num_rollouts=24, num_rollouts_per_batch=4,
                                    move_cutoff=14 if n == 9 else 10, seed=4, record_games=True, resign_thres=0.0)
    tables = []  # (game, ply, visits) of every searched move, as the recorder saw them
    orig = sp.mcts.results

    def spy():
        r = orig()
        info = sp.gb.info()
        for g in range(G):
            tables.append((g, int(info[g, 0]), r["visits"][g].copy()))
        return r
    sp.mcts.results = spy
    while sp.games_finished < G:
        sp.step()
    recs = sp.records
    assert len(recs) >= G
    text = record.dumps(recs)
    assert oracles.ref_record_batch_count(text, n) == len(recs)
    for rec in recs:
        back = oracles.ref_record_roundtrip(json.dumps(rec), n)
        assert back is not None, "the reference's Record::createFromJson rejected a GPU self-play record"
        same(rec, json.loads(back))
        res = rec["result"]
        # the game replays on the REFERENCE board: every recorded move is legal there, in order
        st = oracles.Ref(n)
        from elf_b200.sgf import sgfstr2actions

        moves = sgfstr2actions(res["content"], n)
        for a in moves:
            assert st.forward(int(a))
        assert int(st.info()[0]) - 1 == res["num_move"] == len(moves)
        assert len(res["policies"]) == min(cutoff, res["num_move"])
    # quantisation on real visit tables == the reference's MCTSPolicy::normalize + addMCTSPolicy
    checked = 0
    for g, ply, vis in tables[:: max(1, len(tables) // 40)]:
        acts = np.flatnonzero(vis >= 0)
        if vis[acts].sum() == 0:
            continue
        want = oracles.ref_quantise_policy(acts, vis[acts].astype(np.float32), n)
        np.testing.assert_array_equal(np.asarray(record.quantise_policy(vis, n), np.uint8), want)
        checked += 1
    assert checked > 10
    assert (sp.mcts.errors() == 0).all()
    sp.close()


def test_shim_modules_drive_the_real_engine(monkeypatch):
    """the drop-in modules (elf_b200/shim: `_elf`, `_elfgames_go`) on the device, called the way the
    reference's game.py / GCWrapper call them (the reference tree itself is not on the GPU box;
    tests/test_dropin_shim.py runs its unmodified files on the same modules):
    go.ContextOptions / go.GameOptions -> go.GameContext(co, opt) -> ctx().createSharedMemOptions /
    allocateSharedMem -> AnyP.field()/set(ptr, strides) -> start / wait / step / stop."""
    import os
    import sys

    import torch

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "elf_b200", "shim")
    monkeypatch.syspath_prepend(shim)
    monkeypatch.setenv("ELFB200_BOARD", "9")
    for m in ("_elf", "_elfgames_go"):
        sys.modules.pop(m, None)
    import _elf
    import _elfgames_go as go

    monkeypatch.setattr(go, "BOARD_SIZE", 9)
    n, bs = 9, 16
    co = go.ContextOptions()
    co.num_games, co.batchsize = 8, bs
    ts = co.mcts_options
    ts.num_threads, ts.num_rollouts_per_thread, ts.num_rollouts_per_batch = 1, 16, 4
    ts.persistent_tree, ts.virtual_loss = True, 1
    ts.alg_opt.use_prior, ts.alg_opt.c_puct = True, 1.5
    opt = go.GameOptions()
    opt.mode, opt.use_mcts, opt.move_cutoff, opt.policy_distri_cutoff, opt.resign_thres = "selfplay", True, 10, 4, 0.0
    GC = go.GameContext(co, opt)
    params = GC.getParams()
    assert params["num_action"] == 82 and params["ACTION_PASS"] == -99
    ctx = GC.ctx()
    assert isinstance(ctx, _elf.Context)
    keep = {}
    smem = {}
    for label, keys in (("actor_black", ["s", "pi", "V", "a", "rv"]), ("game_end", []), ("game_start", ["black_ver", "white_ver"])):
        o = ctx.createSharedMemOptions(label, bs if label == "actor_black" else 1)
        o.setTimeout(10)
        sm = ctx.allocateSharedMem(o, keys)
        for k in keys:  # what Allocator._alloc does (utils_elf.py:32-57)
            f = sm[k].field()
            dt = {"float": torch.float32, "int64_t": torch.int64, "int32_t": torch.int32}[f.type_name()]
            t = torch.zeros(f.sz().vec(), dtype=dt).pin_memory()
            sm[k].set(t.data_ptr(), [s_ * t.element_size() for s_ in t.stride()])
            keep[(label, k)] = t
        smem[label] = sm
    ctx.start()
    ends, batches = 0, 0
    for _ in range(4000):
        sm = ctx.wait(0)
        label = sm.getSharedMemOptions().label()
        if label == "actor_black":
            k = sm.effective_batchsize()
            s = keep[(label, "s")][:k]
            assert 0 < k <= bs and set(np.unique(s.numpy())) <= {0.0, 1.0}
            pi, v = oracles.feature_net(s.numpy(), 82)
            keep[(label, "pi")][:k] = torch.from_numpy(pi)
            keep[(label, "V")][:k] = torch.from_numpy(v)
            batches += 1
        elif label == "game_end":
            ends += 1
        ctx.step(_elf.ReplyStatus.SUCCESS)
        if ends >= 8:
            break
    ctx.stop()
    wr = GC.getClient().getGameStats().getWinRateStats()
    assert ends >= 8 and batches > 20 and wr.total_games >= 8


@pytest.mark.skipif(not oracles.have_ref(9), reason="compiled reference (oracle/_ref) not available")
def test_selfplay_on_the_reference_random_streams():
    """SelfPlay(rng="reference") on the device: root noise, D4 code per evaluated leaf, sampled moves and
    the never-resign draw from the reference's own mt19937 streams -- the games of two reference game
    threads (composed from the compiled reference's pieces as GoGameSelfPlay::act orders them), move for
    move, across a game end.  CPU twin on the emulator: tests/test_refstream.py."""
    import torch

    import elf_b200
    from elf_b200.selfplay import SelfPlay

    n, G, moves = 9, 3, 26
    opts = dict(num_rollouts=24, num_rollouts_per_batch=4, virtual_loss=1, persistent_tree=1, c_puct=1.5, komi=7.5)
    eps, alpha, cutoff, thres, ratio, move_cutoff = 0.25, 0.3, 8, 0.05, 0.1, 11
    seeds = np.array([777, 778, 777], np.uint64)
    net = lambda feats, hashes: oracles.feature_net(feats, n * n + 1)  # noqa: E731
    expect = []
    for s in seeds:
        g = oracles.RefRng(n, int(s))
        ref = oracles.RefMcts(n, callback=net, root_epsilon=eps, root_alpha=alpha, rotation_flip=1, seed=g.next(), **opts)
        rc = oracles.RefResign(n, thres, ratio)
        st = oracles.Ref(n)
        played = []
        for _ in range(moves):
            ply = int(st.info()[0])
            r = ref.act(st)
            a = ref.sample(g) if ply <= cutoff else r["best_action"]
            rc.check(r["best_q"], int(st.info()[1]), g)
            assert st.forward(int(a))
            played.append(int(a))
            if st.info()[9] or int(st.info()[0]) >= move_cutoff:
                ref.end_game(st)
                st = oracles.Ref(n)
                rc.reset()
        expect.append(played)

    def actor(batch):
        pi, v = oracles.feature_net(batch["s"].float().cpu().numpy(), n * n + 1)
        return {"pi": torch.from_numpy(pi).to(batch["s"].device), "V": torch.from_numpy(v).to(batch["s"].device)}

    sp = SelfPlay(actor, num_games=G, board_size=n, rng="reference", seed=seeds, policy_distri_cutoff=cutoff,
                  resign_thres=thres, never_resign_ratio=ratio, move_cutoff=move_cutoff, root_epsilon=eps,
                  root_alpha=alpha, rotation_flip=1, **opts)
    got = [[] for _ in range(G)]
    fwd = sp.gb.forward

    def logged(acts):
        for g in range(G):
            got[g].append(int(acts[g]))
        return fwd(acts)

    sp.gb.forward = logged
    for _ in range(moves):
        sp.step()
    assert got == expect
    assert got[0] == got[2] and got[0] != got[1]  # GameOptions::seed: same seed, same game
    assert sp.games_finished >= 2 * G and (sp.mcts.errors() == 0).all()
    sp.close()


@pytest.mark.parametrize("case", range(2))
def test_reference_stream_games_equal_the_golden_reference_games_on_device(case):
    """tests/golden/refstream_games.json (games of the compiled reference's game threads with a seed:
    noise, D4 per leaf, sampled moves, never-resign draw; 9x9 across game ends and 19x19) replayed by
    SelfPlay(rng="reference") on the device -- needs no oracle/_ref on the box"""
    import elf_b200
    from tests.test_refstream_golden import GOLD, run_case

    c = json.load(open(GOLD))[case]
    got = run_case(c, lambda G, n: elf_b200.GoBatch(G, board_size=n), lambda gb, **o: elf_b200.MctsBatch(gb, **o))
    for g, game in enumerate(c["games"]):
        assert got[g] == game["actions"], f"game {g} (seed {game['seed']})"
