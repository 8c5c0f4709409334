"""The kernel SOURCES (elf_b200/csrc/*.cu, board.cuh) executed on the host SIMT emulator
(tests/simt_emu) through the product's own C ABI, against the oracle.

What this proves and what it does not: every lane's arithmetic, the predication of idle lanes, the
warp collectives with partial masks (9x9 packs three games per warp), shared-memory staging and the
node-pool bookkeeping are the code that runs on the GPU, executed here with 32-lane warps whose
collectives complete only when all named lanes arrive (a lane that never arrives, or arrives with a
different operation, aborts the test).  It does not prove anything about timing, inter-warp memory
ordering or hardware behaviour -- the `-m gpu` tests on a B200 are the parity gate; this file keeps
the kernels' logic under test on GPU-less machines and covers paths that have not yet had a GPU run
(G = 1 online mode, parked games, the replay path on the board batch)."""
import numpy as np
import pytest
import torch

from tests import oracles

pytestmark = pytest.mark.timeout(900)


@pytest.fixture(scope="module")
def emu():
    from tests import emu as E

    try:
        E.emu_lib()
    except Exception as e:  # no g++ / ucontext: the emulator is a convenience, not a requirement
        pytest.skip(f"SIMT emulator build unavailable: {e}")
    return E


@pytest.fixture(params=["ascending", "reverse", "random"])
def lane_order(request, emu):
    """order in which the emulator runs the lanes of a warp between two collectives: hardware
    promises none, so results must not depend on it (a missing __syncwarp shows up here)"""
    L = emu.emu_lib()
    L.simt_emu_set_order(["ascending", "reverse", "random"].index(request.param))
    yield request.param
    L.simt_emu_set_order(0)


def fake_actor(search, n):
    def actor(batch):
        h, _, _ = search.leaf_info()
        pi, v = oracles.fakenet(h, n * n + 1)
        assert batch["s"].shape[0] == len(h)
        return {"pi": torch.from_numpy(pi), "V": torch.from_numpy(v)}

    return actor


@pytest.mark.parametrize("n,G", [(9, 5), (19, 3)])
def test_board_kernels(emu, oracle_lib, n, G, lane_order):
    """k_reset / k_step / k_export / k_features: forward verdict, hash, legal mask, info words,
    scores, true eyes and the 18 planes under every D4 code, with illegal and pass moves mixed in;
    9x9 runs 3 games per warp with G = 5 leaving a partially filled warp"""
    gb = emu.emu_batch(G, n)
    os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
    rng = np.random.default_rng(n)
    for t in range(90):
        acts = np.empty(G, np.int32)
        for g, o in enumerate(os_):
            lg = np.flatnonzero(o.legal())
            acts[g] = int(rng.choice(lg)) if len(lg) and rng.random() > 0.05 else n * n
            if rng.random() < 0.05:
                acts[g] = int(rng.integers(n * n))  # possibly illegal
            if rng.random() < 0.03:
                acts[g] = -1  # leave the game untouched
        ok = gb.forward(acts)
        for g, o in enumerate(os_):
            if acts[g] >= 0:
                assert bool(ok[g]) == bool(o.forward(int(acts[g]))), (t, g)
        assert [int(x) for x in gb.getHashCode()] == [o.hash() for o in os_], t
        if t % 6 == 0:
            lm, info, sc, ev = gb.legal_mask(), gb.info(), gb.tt_score(), gb.evaluate(7.5)
            eyes = gb.true_eyes(0)
            for g, o in enumerate(os_):
                assert (lm[g, :-1] == o.legal()).all() and lm[g, -1] == 1
                oi = np.asarray(o.info()).copy()
                oi[8] = 0  # ko_age is not part of the device state
                assert (info[g] == oi).all(), (t, g, info[g], oi)
                assert sc[g] == o.tt_score() and ev[g] == pytest.approx(o.evaluate(7.5))
                assert (eyes[g] == o.true_eyes(int(info[g, 1]))).all()
    d4 = np.arange(G, dtype=np.int32) % 8
    f = gb.features(d4)
    for g, o in enumerate(os_):
        assert (f[g] == o.features(int(d4[g]))).all()
    if oracles.have_ref(n) and lane_order == "ascending":  # GoState::showBoard of the compiled reference
        r = oracles.Ref(n)
        for a in (3, n + 4, n * n, 2 * n + 1):
            r.forward(a)
        gb2 = emu.emu_batch(2, n)
        for a in (3, n + 4, n * n, 2 * n + 1):
            gb2.forward(np.array([a, -1], np.int32))
        assert gb2.showBoard(0) == oracles.ref_show_board(r)
    gb.reset(np.array([1] + [0] * (G - 1), np.uint8))
    assert gb.info()[0, 0] == 1 and gb.getHashCode()[0] == 0 and gb.getHashCode()[1] == os_[1].hash()


@pytest.mark.parametrize("n,G,layout", [(9, 7, 0), (19, 3, 0), (19, 7, 1), (19, 2, 1)])
def test_playout_kernel(emu, oracle_lib, n, G, layout, lane_order):
    """k_playout (incremental safe/atari masks, Bloom-filtered superko, policy pick, checksum):
    to-terminal and steady-state modes, per-game checksums of every intermediate position; layout 1 =
    k_playout2, two board rows per lane, three 19x19 games per warp (G = 7: two full warps and a warp
    with one game; G = 2: a warp with an empty third slot)"""
    gb = emu.emu_batch(G, n)
    gb.set_playout_layout(layout)
    r = gb.playout(1234, first_game_id=50)
    want = oracles.oracle_playout_many(n, 1234, 50, G, lib=oracle_lib)
    np.testing.assert_array_equal(r["chk"], want["chk"])
    np.testing.assert_array_equal(r["plies"], want["plies"])
    np.testing.assert_array_equal(r["score"], want["score"])
    assert r["total_plies"] == want["total_plies"]
    rs = gb.playout_stream(99, first_game_id=7, plies_per_slot=300)
    for s in range(G):
        t, acc, games = oracles.oracle_playout_stream(n, 99, 7, s, G, 300, lib=oracle_lib)
        assert (t, acc, games) == (int(rs["plies"][s]), int(rs["chk"][s]), int(rs["games"][s]))


@pytest.mark.parametrize("n,G,R", [(9, 4, 96), (19, 2, 64)])
def test_search_kernels(emu, oracle_lib, n, G, R, lane_order):
    """k_begin / k_select / k_leaf_features / k_expand / k_backup / k_results / k_advance with tree
    reuse over several moves: root visit counts equal the search restatement's"""
    opts = dict(num_rollouts=R, num_rollouts_per_batch=8, c_puct=1.5, virtual_loss=1, persistent_tree=1)
    gb = emu.emu_batch(G, n)
    mc = emu.EmuSearch(gb, rotation_flip=0, **opts)
    os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
    oms = [oracles.OracleMcts(n, lib=oracle_lib, **opts) for _ in range(G)]
    rng = np.random.default_rng(1)
    for _ in range(6):
        acts = np.array([int(rng.choice(np.flatnonzero(o.legal()))) for o in os_], np.int32)
        assert gb.forward(acts).all()
        for o, a in zip(os_, acts):
            o.forward(int(a))
    actor = fake_actor(mc, n)
    for _ in range(4):
        res = mc.act(actor)
        want = [om.act(o) for om, o in zip(oms, os_)]
        for g in range(G):
            np.testing.assert_array_equal(res["visits"][g], want[g]["visits"])
            assert res["total_visits"][g] == want[g]["total_visits"]
            assert res["root_value"][g] == pytest.approx(want[g]["root_value"], abs=1e-6)
        acts = np.array([w["best_action"] for w in want], np.int32)
        gb.forward(acts)
        mc.advance(acts)
        for o, a in zip(os_, acts):
            o.forward(int(a))
    assert (mc.errors() == 0).all()


def test_leaf_features_of_the_search(emu, oracle_lib):
    """the planes k_leaf_features writes for every leaf (history along the tree path + the game's
    ring, random D4 per evaluation) equal the restatement's extractor on the same position"""
    n, G = 9, 2
    gb = emu.emu_batch(G, n)
    mc = emu.EmuSearch(gb, rotation_flip=1, seed=3, num_rollouts=24, num_rollouts_per_batch=4)
    os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
    rng = np.random.default_rng(8)
    for _ in range(12):
        acts = np.array([int(rng.choice(np.flatnonzero(o.legal()))) for o in os_], np.int32)
        gb.forward(acts)
        for o, a in zip(os_, acts):
            o.forward(int(a))
    seen = []

    def actor(batch):
        h, g, ply = mc.leaf_info()
        seen.append((h.copy(), g.copy(), ply.copy(), mc.leaf_d4.copy(), batch["s"].numpy().copy()))
        pi, v = oracles.fakenet(h, n * n + 1)
        return {"pi": torch.from_numpy(pi), "V": torch.from_numpy(v)}

    mc.search(actor)
    # the first wave's leaves are the roots: planes must be the game's own features under leaf_d4
    h, g, ply, d4, s = seen[0]
    assert len(h) == G and set(d4.tolist()) <= set(range(8))
    for i in range(len(h)):
        o = os_[int(g[i])]
        assert int(h[i]) == o.hash() and int(ply[i]) == int(o.info()[0])
        assert (s[i] == o.features(int(d4[i]))).all()
    # deeper leaves: the side-to-move planes and the stone planes agree with the leaf's ply parity
    for h, g, ply, d4, s in seen[1:]:
        for i in range(len(h)):
            black_to_move = int(ply[i]) % 2 == 1
            assert s[i, 16].all() == black_to_move and s[i, 17].all() == (not black_to_move)
            assert set(np.unique(s[i])) <= {0.0, 1.0}
    assert len({int(x) for _, _, _, d, _ in seen for x in d}) > 1  # the D4 draw varies


def test_online_game_g1_on_the_kernels(emu, oracle_lib):
    """single-game online mode (OnlineGame + GtpConsole) on the real kernels: the G = 1 combination
    with operator moves between searches -- moves equal the restatement's"""
    from elf_b200 import console, online

    n = 9
    opts = dict(num_rollouts=64, num_rollouts_per_batch=8, c_puct=1.5, virtual_loss=1, persistent_tree=1)
    gb = emu.emu_batch(1, n)
    g = online.OnlineGame(gb, emu.EmuSearch(gb, rotation_flip=0, **opts), resign_thres=0.0)
    c = console.GtpConsole(g, fake_actor(g.search, n))
    o = oracles.Oracle(n, oracle_lib)
    om = oracles.OracleMcts(n, lib=oracle_lib, **opts)
    rng = np.random.default_rng(3)
    for t in range(10):
        who = "b" if int(o.info()[1]) == 1 else "w"
        if t % 3 == 2:
            a = int(rng.choice(np.flatnonzero(o.legal())))
            assert c.execute(f"play {who} {online.action2vertex(a, n)}") == "=\n\n"
        else:
            a = om.act(o)["best_action"]
            assert c.execute(f"genmove {who}") == f"= {online.action2vertex(a, n)}\n\n"
        assert o.forward(a)
        assert int(gb.getHashCode()[0]) == o.hash()
    assert "Last move" in c.execute("showboard") and g.seq == 0 and (g.search.errors() == 0).all()
    c.execute("clear_board")
    assert gb.info()[0, 0] == 1 and g.seq == 1


def test_selfplay_loop_with_parked_games_on_the_kernels(emu, oracle_lib):
    """SelfPlay.step with the device-side move choice (k_choose) and a request that parks games:
    parked games are neither searched nor moved, playing games follow the restatement"""
    from elf_b200.selfplay import SelfPlay

    n, G = 9, 4
    opts = dict(num_rollouts=32, num_rollouts_per_batch=4, c_puct=1.5, virtual_loss=1, persistent_tree=1)
    gb = emu.emu_batch(G, n)
    mc = emu.EmuSearch(gb, rotation_flip=0, **opts)
    sp = SelfPlay(fake_actor(mc, n), num_games=G, board_size=n, policy_distri_cutoff=0, never_resign_ratio=1.0,
                  board=gb, search=mc)
    assert sp.set_request(1, -1, 0.05, num_game_thread_used=3) == "update_model"
    os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
    oms = [oracles.OracleMcts(n, lib=oracle_lib, **opts) for _ in range(G)]
    for _ in range(3):
        want = [oms[g].act(os_[g])["best_action"] for g in range(3)]
        assert sp.step() == 3
        for g in range(3):
            assert os_[g].forward(want[g])
        h = gb.getHashCode()
        assert [int(h[g]) for g in range(3)] == [os_[g].hash() for g in range(3)] and int(h[3]) == 0
    assert gb.info()[:, 0].tolist() == [4, 4, 4, 1] and (mc.errors() == 0).all()


def test_replay_batch_on_the_board_kernels(emu, oracle_lib):
    """ReplayBatch on the real board batch (k_reset / k_step with untouched games / k_features with
    per-sample D4) equals ReplayBatch on oracle boards"""
    from elf_b200 import record, replay
    from tests.test_request_protocol import Boards

    n, B = 9, 5
    rng = np.random.default_rng(6)
    recs = []
    for i in range(3):
        o = oracles.Oracle(n, oracle_lib)
        r = record.GameRecorder(n, i, 8)
        for t in range(25 + 7 * i):
            lg = np.flatnonzero(o.legal())
            a = int(rng.choice(lg)) if len(lg) else n * n
            row = np.full(n * n + 1, -1, np.int32)
            row[rng.choice(n * n + 1, 10, replace=False)] = rng.integers(1, 99, 10)
            r.on_move(int(o.info()[0]), a, row, 0.0)
            o.forward(a)
        recs.append(r.finish(1.0 if i % 2 else -1.0, False, model_ver=i))
    a_ = replay.ReplayBatch(B, board_size=n, num_future_actions=2, board=emu.emu_batch(B, n))
    b_ = replay.ReplayBatch(B, board_size=n, num_future_actions=2, board=Boards(B, oracle_lib))
    a_.add_records(recs)
    b_.add_records(recs)
    picks = [(0, 0, 1), (1, 30, 6), (2, 37, 3), (0, 23, 7), (2, 5, 0)]
    x, y = a_.sample(picks), b_.sample(picks)
    for k in x:
        np.testing.assert_array_equal(x[k], y[k])
    # planes written by the feature kernel straight into the caller's tensor
    dst = torch.full((B, 18, n, n), -1.0)
    z = a_.sample(picks, s_out=dst)
    assert z["s"] is dst
    np.testing.assert_array_equal(dst.numpy(), y["s"])


@pytest.mark.parametrize("n,G", [(9, 7), (19, 3)])
def test_replay_kernel(emu, oracle_lib, n, G, lane_order):
    """k_replay (one launch forwards every game's own move list from the empty board) leaves exactly
    the state that the same moves leave through k_step -- position, info words, legal rows, the
    8-position history seen by the feature kernel and the superko record (checked by playing on)"""
    rng = np.random.default_rng(n)
    lists, os_ = [], []
    for g in range(G):
        o = oracles.Oracle(n, oracle_lib)
        mv = []
        for _ in range(0 if g == 1 else int(rng.integers(1, 70 if n == 9 else 200))):
            lg = np.flatnonzero(o.legal())
            a = int(rng.choice(lg)) if len(lg) and rng.random() > 0.04 else n * n
            if rng.random() < 0.05:
                a = int(rng.integers(n * n))  # possibly refused: skipped, the list goes on
            mv.append(a)
            o.forward(a)
        lists.append(mv)
        os_.append(o)
    gb = emu.emu_batch(G, n)
    gb.forward(np.full(G, 3, np.int32))  # state that the replay has to wipe
    gb.replay(lists)
    ref = emu.emu_batch(G, n)
    for t in range(max(len(m) for m in lists)):
        ref.forward(np.array([m[t] if t < len(m) else -1 for m in lists], np.int32))
    assert [int(h) for h in gb.getHashCode()] == [o.hash() for o in os_]
    np.testing.assert_array_equal(gb.info(), ref.info())
    np.testing.assert_array_equal(gb.stones(), ref.stones())
    np.testing.assert_array_equal(gb.legal_mask(), ref.legal_mask())
    d4 = np.arange(G, dtype=np.int32) % 8
    np.testing.assert_array_equal(gb.features(d4), ref.features(d4))
    for _ in range(40):
        acts = np.array([int(rng.choice(np.flatnonzero(o.legal()))) if o.legal().any() and not o.terminated() else n * n
                         for o in os_], np.int32)
        ok = gb.forward(acts)
        for g, o in enumerate(os_):
            assert bool(ok[g]) == bool(o.forward(int(acts[g])))
        assert [int(h) for h in gb.getHashCode()] == [o.hash() for o in os_]
    with pytest.raises(Exception, match="stride"):
        gb.replay([[0] * (2 * n * n + 1)] * G)


def test_wait_step_pump_on_the_kernels(emu):
    """the host path of tests/test_gpu_compat.py::test_wait_step_pump_plays_games (no request ever
    set, host-memory SharedMems, a small network answering the actor_black batches) with the
    kernels on the emulator: games are played to the move cutoff and restarted"""
    from elf_b200 import compat
    from elf_b200.model import Actor, PolicyValueNet
    from elf_b200.selfplay import SelfPlay

    torch.manual_seed(0)
    n, G, BS = 9, 6, 8
    net = Actor(PolicyValueNet(n, num_block=1, dim=8), batchsize=BS, dtype=torch.float32, channels_last=False)
    gb = emu.emu_batch(G, n)
    mc = emu.EmuSearch(gb, num_rollouts=8, num_rollouts_per_batch=4, rotation_flip=1, seed=3)
    sp = SelfPlay(None, num_games=G, board_size=n, policy_distri_cutoff=0, move_cutoff=5, seed=3, board=gb, search=mc)
    GC = compat.GameContext(compat.SelfPlayEngine(sp), batchsize=BS)
    ctx = GC.ctx()
    keys = ["s", "pi", "V", "a", "rv"]
    opts = ctx.createSharedMemOptions("actor_black", BS)
    bufs = {}
    for _ in range(2):
        sm = ctx.allocateSharedMem(opts, keys)
        b = {}
        for k in keys:
            f = sm[k].field()
            dt = {"float": torch.float32, "int64_t": torch.int64, "int32_t": torch.int32}[f.type_name()]
            b[k] = torch.zeros(*f.sz().vec(), dtype=dt)
            sm[k].set(b[k].data_ptr(), [i * b[k].element_size() for i in b[k].stride()])
        bufs[sm.getSharedMemOptions().idx()] = b
    ctx.start()
    batches = 0
    while sp.games_finished < G and batches < 400:
        sm = ctx.wait()
        k = sm.effective_batchsize()
        assert 0 < k <= BS and sm.getSharedMemOptions().label() == "actor_black"
        b = bufs[sm.getSharedMemOptions().idx()]
        ind = b["s"][:k, 16:18].reshape(k, 2, -1)
        assert ((ind.sum(2) == n * n).sum(1) == 1).all()  # exactly one side-to-move plane is set
        out = net({"s": b["s"][:k]})
        b["pi"][:k].copy_(out["pi"])
        b["V"][:k].copy_(out["V"])
        ctx.step()
        batches += 1
    ctx.stop()
    assert sp.games_finished >= G and sp.moves_played >= 4 * G and (mc.errors() == 0).all()
    assert GC.getClient().getGameStats().getWinRateStats().total_games == sp.games_finished


def test_online_engine_pump_on_the_kernels(emu, oracle_lib):
    """mode == "online" through compat.Context with the kernels on the emulator: human_actor asks
    for an action, ACTION_SKIP starts a search whose waves (8 leaves) arrive as actor_black batches of
    <= 3, and the move played is the restatement's"""
    from elf_b200 import compat, online

    n = 9
    opts = dict(num_rollouts=32, num_rollouts_per_batch=8, c_puct=1.5, virtual_loss=1, persistent_tree=1)
    gb = emu.emu_batch(1, n)
    search = emu.EmuSearch(gb, rotation_flip=0, **opts)
    g = online.OnlineGame(gb, search)
    GC = compat.GameContext(compat.OnlineEngine(g), batchsize=3)
    ctx = GC.ctx()
    bufs = {}
    for label, keys, bs in (("human_actor", ["s", "pi", "a", "V"], 1), ("actor_black", ["s", "pi", "V", "a", "rv"], 3)):
        sm = ctx.allocateSharedMem(ctx.createSharedMemOptions(label, bs), keys)
        b = {}
        for k in keys:
            f = sm[k].field()
            dt = {"float": torch.float32, "int64_t": torch.int64, "int32_t": torch.int32}[f.type_name()]
            b[k] = torch.zeros(*f.sz().vec(), dtype=dt)
            sm[k].set(b[k].data_ptr(), [i * b[k].element_size() for i in b[k].stride()])
        bufs[label] = b
    o = oracles.Oracle(n, oracle_lib)
    om = oracles.OracleMcts(n, lib=oracle_lib, **opts)
    script = [online.vertex2action("E5", n), online.SA_SKIP, online.vertex2action("C3", n), online.SA_SKIP, online.SA_SKIP]
    ctx.start()
    chunks = []
    for cmd in script:
        sm = ctx.wait()
        assert sm.getSharedMemOptions().label() == "human_actor" and sm.effective_batchsize() == 1
        assert (bufs["human_actor"]["s"][0].numpy() == o.features(0)).all()  # the operator sees the position
        bufs["human_actor"]["a"][0] = cmd
        ctx.step()
        if cmd != online.SA_SKIP:
            assert o.forward(cmd)
            continue
        want = om.act(o)["best_action"]
        while GC._engine.next_label() == "actor_black":
            sm = ctx.wait()
            k = sm.effective_batchsize()
            chunks.append(k)
            # the leaves of a wave arrive in slot order; the fake net needs their hashes
            h, _, _ = search.leaf_info()
            base = GC._engine._wave["off"] - k
            pi, v = oracles.fakenet(h[base:base + k], n * n + 1)
            bufs["actor_black"]["pi"][:k] = torch.from_numpy(pi)
            bufs["actor_black"]["V"][:k] = torch.from_numpy(v)
            ctx.step()
        assert o.forward(want) and int(gb.getHashCode()[0]) == o.hash()
    ctx.stop()
    assert max(chunks) == 3 and len(chunks) > 12 and (search.errors() == 0).all()
    assert GC.getGame(0).getNextPlayer() in "BW" and "Last move" in GC.getGame(0).showBoard()


def test_search_option_fuzz(emu, oracle_lib):
    """random search options (rollouts not a multiple of the batch, batch 1..16, virtual loss 0..3,
    tree reuse on/off, priors off, FPU switches, pass rules, komi), random openings, 1..4 games,
    terminated games left inactive: root visit tables equal the restatement's in every case"""
    n = 9
    rng = np.random.default_rng(7)
    for case in range(8):
        opts = dict(
            num_rollouts=int(rng.integers(8, 90)), num_rollouts_per_batch=int(rng.integers(1, 17)),
            virtual_loss=int(rng.integers(0, 4)), persistent_tree=int(rng.integers(0, 2)),
            c_puct=float(rng.choice([0.5, 0.85, 1.5, 2.5, 5.0])), unexplored_q_zero=int(rng.integers(0, 2)),
            root_unexplored_q_zero=int(rng.integers(0, 2)), ply_pass_enabled=int(rng.choice([0, 30, 70])),
            remove_pass_if_dangerous=int(rng.integers(0, 2)), komi=float(rng.choice([5.5, 6.5, 7.5])),
            use_prior=int(rng.random() > 0.15))
        G, open_plies = int(rng.integers(1, 5)), int(rng.integers(0, 75))
        emu.emu_lib().simt_emu_set_order(case % 3)
        gb = emu.emu_batch(G, n)
        mc = emu.EmuSearch(gb, rotation_flip=0, **opts)
        os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
        oms = [oracles.OracleMcts(n, lib=oracle_lib, **opts) for _ in range(G)]
        for _ in range(open_plies):
            acts = np.array([int(rng.choice(np.flatnonzero(o.legal()))) if o.legal().any() and not o.terminated() else n * n
                             for o in os_], np.int32)
            gb.forward(acts)
            for o, a in zip(os_, acts):
                o.forward(int(a))
        actor = fake_actor(mc, n)
        for mv in range(3):
            live = np.array([not o.terminated() for o in os_])
            if not live.any():
                break
            res = mc.act(actor, active=live.astype(np.uint8))
            acts = np.full(G, -1, np.int32)
            for g in np.flatnonzero(live):
                w = oms[g].act(os_[g])
                np.testing.assert_array_equal(res["visits"][g], w["visits"], err_msg=f"case {case} move {mv} {opts}")
                assert res["total_visits"][g] == w["total_visits"]
                acts[g] = w["best_action"]
            gb.forward(acts)
            mc.advance(acts)
            for o, a in zip(os_, acts):
                if a >= 0:
                    o.forward(int(a))
        assert (mc.errors() == 0).all(), (case, opts)
    emu.emu_lib().simt_emu_set_order(0)


def test_two_model_pump_on_the_kernels(emu):
    """host path of tests/test_gpu_compat.py::test_two_models_route_to_actor_black_and_actor_white
    with the kernels on the emulator: two trees over one board batch, leaves of black-to-move games
    under actor_black, of white-to-move games under actor_white"""
    from elf_b200 import compat
    from elf_b200.model import Actor, PolicyValueNet
    from elf_b200.selfplay import SelfPlay

    torch.manual_seed(1)
    n, G, BS = 9, 4, 16
    nets = {lab: Actor(PolicyValueNet(n, num_block=1, dim=8), batchsize=BS, dtype=torch.float32, channels_last=False)
            for lab in ("actor_black", "actor_white")}
    gb = emu.emu_batch(G, n)
    opts = dict(num_rollouts=8, num_rollouts_per_batch=4, rotation_flip=0)
    sp = SelfPlay(nets["actor_black"], actor_white=nets["actor_white"], num_games=G, board_size=n, policy_distri_cutoff=0,
                  move_cutoff=6, seed=2, board=gb, search=emu.EmuSearch(gb, **opts), search_white=emu.EmuSearch(gb, **opts))
    GC = compat.GameContext(compat.SelfPlayEngine(sp), batchsize=BS)
    ctx = GC.ctx()
    keys = ["s", "pi", "V", "a", "rv"]
    bufs, counts = {}, {"actor_black": 0, "actor_white": 0}
    for lab in counts:
        o = ctx.createSharedMemOptions(lab, BS)
        sm = ctx.allocateSharedMem(o, keys)
        b = {}
        for k in keys:
            f = sm[k].field()
            dt = {"float": torch.float32, "int64_t": torch.int64, "int32_t": torch.int32}[f.type_name()]
            b[k] = torch.zeros(*f.sz().vec(), dtype=dt)
            sm[k].set(b[k].data_ptr(), [i * b[k].element_size() for i in b[k].stride()])
        bufs[sm.getSharedMemOptions().idx()] = b
    ctx.start()
    it = 0
    while sp.games_finished < G and it < 300:
        sm = ctx.wait()
        lab, k = sm.getSharedMemOptions().label(), sm.effective_batchsize()
        b = bufs[sm.getSharedMemOptions().idx()]
        _, games, _ = GC._engine._wave["mc"].leaf_info()  # the wave's leaves belong to games whose ROOT mover matches the label
        root_black = gb.info()[games, 1] == 1
        assert root_black.all() if lab == "actor_black" else (~root_black).all()
        out = nets[lab]({"s": b["s"][:k]})
        b["pi"][:k].copy_(out["pi"])
        b["V"][:k].copy_(out["V"])
        ctx.step()
        counts[lab] += k
        it += 1
    ctx.stop()
    assert counts["actor_black"] > 0 and counts["actor_white"] > 0 and sp.games_finished >= G
    assert (sp.mcts.errors() == 0).all() and (sp.mcts2.errors() == 0).all()


@pytest.mark.parametrize("two_models", [False, True])
def test_policy_only_colour_on_the_kernels(emu, oracle_lib, two_models):
    """white_use_policy_network_only (GoGameSelfPlay::act -> actPolicyOnly): white plays the arg-max
    of the network policy over its legal moves without searching (one root evaluation at most), black
    searches as usual; with one shared tree white's root is usually already expanded by black's search"""
    from elf_b200.selfplay import SelfPlay

    n, G = 9, 3
    opts = dict(num_rollouts=32, num_rollouts_per_batch=4, c_puct=1.5, virtual_loss=1, persistent_tree=1)
    gb = emu.emu_batch(G, n)
    mc = emu.EmuSearch(gb, rotation_flip=0, **opts)
    mc2 = emu.EmuSearch(gb, rotation_flip=0, **opts) if two_models else None
    calls = []

    def make_actor(search, tag):
        inner = fake_actor(search, n)

        def actor(batch):
            calls.append((tag, batch["s"].shape[0]))
            return inner(batch)

        return actor

    sp = SelfPlay(make_actor(mc, "b"), actor_white=make_actor(mc2, "w") if two_models else None, num_games=G, board_size=n,
                  policy_distri_cutoff=0, never_resign_ratio=1.0, white_use_policy_network_only=True, record_games=True,
                  board=gb, search=mc, search_white=mc2)
    os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
    oms = [oracles.OracleMcts(n, lib=oracle_lib, **opts) for _ in range(G)]
    for mv in range(6):
        black = mv % 2 == 0
        want = []
        for g, o in enumerate(os_):
            if black:
                want.append(oms[g].act(o)["best_action"])
            else:
                pi, _ = oracles.fakenet(np.array([o.hash()], np.uint64), n * n + 1)
                legal = np.append(o.legal().astype(bool), True)
                want.append(int(np.where(legal, pi[0], -1.0).argmax()))
        del calls[:]
        assert sp.step() == G
        if not black:  # at most one root evaluation per game, nothing else
            assert sum(k for _, k in calls) <= G and all(t == ("w" if two_models else "b") for t, _ in calls)
        for o, a in zip(os_, want):
            assert o.forward(a)
        assert [int(h) for h in gb.getHashCode()] == [o.hash() for o in os_], (mv, want)
    # records: MCTS policies only for the searched (black) moves while ply <= cutoff (0 here: none), values for all
    sp.move_cutoff = 1
    sp.step()
    assert len(sp.records) == G and all(len(r["result"]["values"]) == 7 for r in sp.records)


def test_game_context_from_options_on_the_kernels(emu):
    """compat.game_context(ContextOptions, GameOptions) -> engine -> wait/step pump, with the engine
    built on the emulated kernels: the option mapping produces a search that actually runs"""
    from elf_b200 import compat, lib as _l
    from elf_b200.selfplay import SelfPlay

    n = 9
    co, opt = compat.ContextOptions(), compat.GameOptions()
    co.num_games, co.batchsize = 3, 8
    m = co.mcts_options
    m.num_threads, m.num_rollouts_per_thread, m.num_rollouts_per_batch, m.virtual_loss, m.persistent_tree = 2, 8, 4, 1, True
    m.alg_opt.c_puct = 1.5
    opt.mode, opt.policy_distri_cutoff, opt.move_cutoff = "selfplay", 0, 4
    built = {}

    def factory(**kw):
        fields = {f[0] for f in _l.MctsOptions._fields_}
        gb = emu.emu_batch(kw["num_games"], kw["board_size"])
        mk = {k: v for k, v in kw.items() if k in fields and k != "seed"}
        built["search"] = emu.EmuSearch(gb, **mk)
        return SelfPlay(board=gb, search=built["search"], **kw)

    GC = compat.game_context(co, opt, board_size=n, factories={"selfplay": factory})
    assert built["search"].options.num_rollouts == 16 and built["search"].waves_per_move == 4
    assert built["search"].options.c_puct == 1.5 and built["search"].options.komi == 7.5
    ctx = GC.ctx()
    sm = ctx.allocateSharedMem(ctx.createSharedMemOptions("actor_black", 8), ["s", "pi", "V", "a", "rv"])
    bufs = {}
    for k in ("s", "pi", "V", "a", "rv"):
        f = sm[k].field()
        dt = {"float": torch.float32, "int64_t": torch.int64, "int32_t": torch.int32}[f.type_name()]
        bufs[k] = torch.zeros(*f.sz().vec(), dtype=dt)
        sm[k].set(bufs[k].data_ptr(), [i * bufs[k].element_size() for i in bufs[k].stride()])
    ctx.start()
    sp = GC._engine.sp
    it = 0
    while sp.games_finished < 3 and it < 200:
        s = ctx.wait()
        k = s.effective_batchsize()
        bufs["pi"][:k] = torch.rand(k, n * n + 1)
        bufs["V"][:k] = 0.0
        ctx.step()
        it += 1
    ctx.stop()
    assert sp.games_finished >= 3 and len(sp.records) == sp.games_finished  # selfplay mode keeps the records
    assert sp.records[0]["request"]["vers"]["mcts_opt"]["num_rollouts_per_thread"] == 16


@pytest.mark.parametrize("n", [9, 19])
def test_fast_feature_formats_async_waves_prune_and_mismatch(emu, n):
    """round-2 kernel paths on the emulator: 16-bit NHWC leaf features equal the float32 ones, waves
    without a host read-back (fixed grids, device-side leaf count) give the same search, a short node
    pool prunes least-visited root subtrees instead of dropping the tree, a stale root is reported"""
    G, R, B = 4, 16, 4
    opts = dict(num_rollouts=R, num_rollouts_per_batch=B, rotation_flip=1, seed=7)

    def make(**kw):
        gb = emu.emu_batch(G, n)
        rng = np.random.default_rng(2)
        os_ = [oracles.Oracle(n) for _ in range(G)]
        for _ in range(9):  # more than 8 plies: the history gather crosses from the tree into the ring
            acts = np.array([int(rng.choice(np.flatnonzero(o.legal()))) for o in os_], np.int32)
            for o, a in zip(os_, acts):
                o.forward(int(a))
            assert gb.forward(acts).all()
        return gb, emu.EmuSearch(gb, **opts, **kw)

    def actor_for(mc, log=None):
        def actor(batch):
            h, _, _ = mc.leaf_info()
            key = "s" if "s" in batch else "s_nhwc"
            x = batch[key]
            if log is not None:
                xx = x[: len(h)].float()
                log.append(xx.numpy().copy() if key == "s" else xx.permute(0, 3, 1, 2)[:, :18].numpy().copy())
                if key != "s":
                    assert (xx[..., 18:] == 0).all()
            pi, v = oracles.fakenet(h, n * n + 1)
            P, V = torch.zeros(x.shape[0], n * n + 1), torch.zeros(x.shape[0])
            P[: len(h)], V[: len(h)] = torch.from_numpy(pi), torch.from_numpy(v)
            return {"pi": P, "V": V}
        return actor

    gb0, m0 = make()
    log0 = []
    r0 = m0.act(actor_for(m0, log0))
    for fmt, cpad in (("f16", 24), ("bf16", 32)):
        gb1, m1 = make(feature_format=fmt, cpad=cpad)
        gb1.set_feature_store(1 if fmt == "f16" else 0)  # staged + bulk store / direct 16-byte stores
        log1 = []
        r1 = m1.act(actor_for(m1, log1))
        assert len(log0) == len(log1)
        for a, b in zip(log0, log1):
            np.testing.assert_array_equal(a, b)
        np.testing.assert_array_equal(r0["visits"], r1["visits"])
    # asynchronous waves
    gb2, m2 = make()
    act2 = actor_for(m2)
    m2.begin_move()
    for _ in range(m2.waves_per_move):
        s = m2.select(wait=False)
        assert s.shape[0] == m2.max_leaves
        m2._n = m2.leaf_count()      # the fake net needs the hashes of the claimed leaves only
        rep = act2({"s": s})
        m2.expand_backup(rep["pi"], rep["V"])
    r2 = m2.results()
    np.testing.assert_array_equal(r0["visits"], r2["visits"])
    assert m2.eval_count() == m0.eval_count()
    # fully asynchronous waves (no count on the host at all: fixed grids everywhere) with a net that
    # reads the planes, against the same net through the synchronous path
    def plane_actor(batch):
        x = batch["s"] if "s" in batch else batch["s_nhwc"].float().permute(0, 3, 1, 2)[:, :18]
        pi, v = oracles.feature_net(x.float().numpy(), n * n + 1)
        return {"pi": torch.from_numpy(pi), "V": torch.from_numpy(v)}

    gb4, m4 = make()
    r4 = m4.act(plane_actor)
    gb5, m5 = make(feature_format="f16")
    m5.begin_move()
    for _ in range(m5.waves_per_move):
        rep = plane_actor({"s_nhwc": m5.select(wait=False)})
        m5.expand_backup(rep["pi"], rep["V"])
    r5 = m5.results()
    np.testing.assert_array_equal(r4["visits"], r5["visits"])
    assert m5.eval_count() == m4.eval_count() and (m5.errors() == 0).all()
    # stale root: the board moves without advance()
    a = r0["best_action"]
    assert gb0.forward(a).all()
    with pytest.raises(Exception, match="Root state is not the same"):
        m0.act(actor_for(m0))
    r = m0.act(actor_for(m0))
    assert (r["total_visits"] == R - B).all() and m0.errors()[0] == G
    # short pool: prune, never overflow
    gb3 = emu.emu_batch(G, n)
    m3 = emu.EmuSearch(gb3, num_rollouts=R, num_rollouts_per_batch=B, rotation_flip=0, nodes_per_game=R + 6)
    act3 = actor_for(m3)
    for _ in range(6):
        r = m3.act(act3)
        assert ((r["total_visits"] == R - B) | (r["total_visits"] >= R)).all()
        assert gb3.forward(r["best_action"]).all()
        m3.advance(r["best_action"])
    e = m3.errors()
    assert e[0] == 0 and e[1] == 0 and e[2] == 0 and e[3] > 0, e


@pytest.mark.parametrize("n,G", [(9, 4), (19, 3)])
def test_darkforest_features_vs_reference(emu, n, G):
    """k_features_df == the compiled reference's BoardFeature::extract (25 DarkForest planes: liberty
    classes, simple ko, stones, exp(last_placed - ply) history, L1 distance maps, side indicators) under
    every D4 code, on positions with captures and kos; elfb200_replay keeps the placement plies too"""
    if not oracles.have_ref(n):
        pytest.skip("oracle/_ref not built")
    gb = emu.emu_batch(G, n)
    refs = [oracles.Ref(n) for _ in range(G)]
    rng = np.random.default_rng(n)
    lists = [[] for _ in range(G)]
    for t in range(70 if n == 9 else 170):
        acts = np.empty(G, np.int32)
        for g, r in enumerate(refs):
            idx = np.flatnonzero(r.legal() & (1 - r.true_eyes(int(r.info()[1]))))
            acts[g] = int(rng.choice(idx)) if len(idx) else n * n
            assert r.forward(acts[g])
            lists[g].append(int(acts[g]))
        assert gb.forward(acts).all()
        if t % 13 == 5 or t > (60 if n == 9 else 160):
            d4 = rng.integers(0, 8, G).astype(np.int32)
            got = gb.features_df(d4)
            for g, r in enumerate(refs):
                want = r.features_df(int(d4[g]))
                for pl in range(25):
                    np.testing.assert_array_equal(got[g, pl], want[pl], err_msg=f"plane {pl} game {g} ply {t} d4 {d4[g]}")
    assert sum(int(r.info()[2] + r.info()[3]) for r in refs) > 0  # captures happened
    gb2 = emu.emu_batch(G, n)
    gb2.replay(lists)
    np.testing.assert_array_equal(gb2.features_df(), gb.features_df())


def test_expand_half_size_sort_network_on_late_positions(emu, oracle_lib):
    """19x19 positions past the opening have at most 256 candidates: k_expand compacts them and sorts with
    the half-size network.  Same priors, same visits as the search restatement; the boundary (a position
    with more than 256 legal moves next to ones with fewer) is crossed inside one batch."""
    n, G = 19, 3
    opts = dict(num_rollouts=24, num_rollouts_per_batch=4, c_puct=1.5, virtual_loss=1, persistent_tree=1)
    gb = emu.emu_batch(G, n)
    mc = emu.EmuSearch(gb, rotation_flip=0, **opts)
    os_ = [oracles.Oracle(n, oracle_lib) for _ in range(G)]
    oms = [oracles.OracleMcts(n, lib=oracle_lib, **opts) for _ in range(G)]
    rng = np.random.default_rng(8)
    plies = [150, 104, 20]  # ~215 legal moves, around the 256 boundary, > 256 (full network)
    for t in range(max(plies)):
        acts = np.full(G, -1, np.int32)
        for g, o in enumerate(os_):
            if t < plies[g]:
                idx = np.flatnonzero(o.legal() & (1 - o.true_eyes(int(o.info()[1]))))
                acts[g] = int(rng.choice(idx)) if len(idx) else n * n
                o.forward(int(acts[g]))
        gb.forward(acts)
    counts = [int(o.legal().sum()) for o in os_]
    assert counts[0] < 256 and counts[2] > 256, counts
    actor = fake_actor(mc, n)
    for _ in range(2):
        res = mc.act(actor)
        pri = mc.root_priors()
        want = [om.act(o) for om, o in zip(oms, os_)]
        for g in range(G):
            np.testing.assert_array_equal(res["visits"][g], want[g]["visits"])
            w = np.where(want[g]["visits"] >= 0, want[g]["prior"], -1.0).astype(np.float32)
            np.testing.assert_array_equal(pri[g], w)  # priors bit-identical (sorted order drives the float sum)
        acts = np.array([w["best_action"] for w in want], np.int32)
        gb.forward(acts)
        mc.advance(acts)
        for o, a in zip(os_, acts):
            o.forward(int(a))
    assert (mc.errors() == 0).all()


@pytest.mark.parametrize("name", ["9_noprior_ties", "9_rounding_ties", "9_superko_in_tree", "9_equal_priors",
                                  "19_equal_priors"])
def test_puct_ties_resolve_in_the_reference_container_order(emu, name, lane_order):
    """k_select's uct_tie_break: exactly equal PUCT scores (no prior term; priors lost in the rounding of
    q) go to the first tied edge in the order of the reference's unordered_map, also when that edge lies
    beyond the scanned prefix (the node is scanned in full from then on) -- root visit tables equal the
    COMPILED reference search's, move after move (twin of test_gpu_mcts.py::test_gpu_search_vs_reference).
    9_superko_in_tree: a recapture two plies below the root repeats a position of the game -- a terminal
    node inside the tree; the 9x9 search used to miss such a repetition when the move captured and the
    matching record was scanned by a lane beyond the board's rows (found by scripts/emu_fuzz_streams.py).
    *_equal_priors: a net with bit-equal probabilities among the legal moves (std_sort_ties, k_expand<N, true>);
    priors bit-identical too"""
    from tests.test_mcts_oracle_vs_ref import SCENARIOS, ref_mcts, scenario_net, scenario_openings, search_options

    sc = SCENARIOS[name]
    n, G = sc["n"], sc["G"]
    if not oracles.have_ref(n):
        pytest.skip("compiled reference (oracle/_ref) not available")
    rng = np.random.default_rng(5 + n)
    gb = emu.emu_batch(G, n)
    states = [oracles.Ref(n) for _ in range(G)]
    fixed = scenario_openings(sc)
    for t in range(sc["open_plies"]):
        acts = np.empty(G, np.int32)
        for g, s in enumerate(states):
            idx = np.flatnonzero(s.legal())
            acts[g] = int(fixed[g][t]) if fixed is not None else int(rng.choice(idx))
            assert s.forward(acts[g])
        assert gb.forward(acts).all()
    mc = emu.EmuSearch(gb, rotation_flip=0, **search_options(sc), **sc["opts"])
    refs = [ref_mcts(sc) for _ in range(G)]
    net = scenario_net(sc)
    if net is None:
        actor = fake_actor(mc, n)
    else:
        def actor(batch):
            pi, v = net(None, mc.leaf_info()[0])
            return {"pi": torch.from_numpy(pi), "V": torch.from_numpy(v)}
    for mv in range(sc["moves"]):
        res = mc.act(actor)
        pri = mc.root_priors()
        acts = np.empty(G, np.int32)
        for g in range(G):
            rr = refs[g].act(states[g])
            np.testing.assert_array_equal(res["visits"][g], rr["visits"], err_msg=f"move {mv} game {g}")
            has = rr["visits"] >= 0
            np.testing.assert_array_equal(pri[g][has], rr["prior"][has], err_msg=f"priors, move {mv} game {g}")
            assert res["total_visits"][g] == rr["total_visits"] and res["best_action"][g] == rr["best_action"]
            assert res["root_value"][g] == np.float32(rr["root_value"]) and abs(res["best_q"][g] - rr["best_q"]) < 1e-5
            acts[g] = rr["best_action"]
            assert states[g].forward(acts[g])
        assert gb.forward(acts).all()
        mc.advance(acts)
    assert (mc.errors() == 0).all(), mc.errors()
    assert mc.eval_count() == sum(c.num_evals() for c in refs)


@pytest.mark.parametrize("n,quant", [(9, 16), (9, 256), (19, 256)])
def test_equal_priors_follow_std_sort(emu, n, quant, lane_order):
    """k_expand<N, true> (search option std_sort_ties): a reply with bit-equal probabilities is put in the
    order libstdc++'s std::sort leaves it in (stdsort.cuh) before the legality filter, as
    MCTSActor::pi2response does; root visit tables, priors and container order then equal the COMPILED
    reference's on networks full of equal values (what half precision produces)"""
    from tests.test_mcts_oracle_vs_ref import quantised_fakenet

    if not oracles.have_ref(n):
        pytest.skip("compiled reference (oracle/_ref) not available")
    rng = np.random.default_rng(100 * n + quant)
    net = quantised_fakenet(n, quant)
    for case in range(3 if n == 9 else 1):
        opts = dict(num_rollouts=int(rng.integers(20, 64 if n == 9 else 40)), num_rollouts_per_batch=int(rng.integers(1, 9)),
                    virtual_loss=int(rng.integers(0, 3)), persistent_tree=1, c_puct=float(rng.choice([0.5, 1.5])),
                    ply_pass_enabled=int(rng.choice([0, 40])))
        G = 2
        gb = emu.emu_batch(G, n)
        refs = [oracles.Ref(n) for _ in range(G)]
        rms = [oracles.RefMcts(n, callback=net, **opts) for _ in range(G)]
        mc = emu.EmuSearch(gb, rotation_flip=0, std_sort_ties=1, **opts)

        def actor(batch):
            h, _, _ = mc.leaf_info()
            pi, v = net(None, h)
            return {"pi": torch.from_numpy(pi), "V": torch.from_numpy(v)}

        for _ in range(int(rng.integers(0, 60 if n == 9 else 150))):
            acts = np.array([int(rng.choice(np.flatnonzero(r.legal()))) for r in refs], np.int32)
            assert gb.forward(acts).all() and all(r.forward(int(a)) for r, a in zip(refs, acts))
        for mv in range(3):
            res, pri = mc.act(actor), mc.root_priors()
            acts = np.empty(G, np.int32)
            for g in range(G):
                w = rms[g].act(refs[g])
                np.testing.assert_array_equal(res["visits"][g], w["visits"], err_msg=f"case {case} move {mv} game {g}")
                has = w["visits"] >= 0
                np.testing.assert_array_equal(pri[g][has], w["prior"][has])
                assert res["best_action"][g] == w["best_action"]
                acts[g] = w["best_action"]
                assert refs[g].forward(int(acts[g]))
            assert gb.forward(acts).all()
            mc.advance(acts)
        assert (mc.errors() == 0).all(), mc.errors()


def test_async_leaf_count_then_leaf_info(emu):
    """the asynchronous wave from Python: select(wait=False) -> leaf_count() -> leaf_info() (the hashes of
    exactly the counted leaves) -> fake net -> expand_backup checked against the known count; root tables
    equal the synchronous search's"""
    n, G = 9, 4
    opts = dict(num_rollouts=40, num_rollouts_per_batch=5, virtual_loss=1, persistent_tree=1, c_puct=1.5)

    def make():
        gb = emu.emu_batch(G, n)
        rng = np.random.default_rng(4)
        for _ in range(12):
            lm = gb.legal_mask()[:, :-1]
            assert gb.forward(np.array([int(rng.choice(np.flatnonzero(r))) for r in lm], np.int32)).all()
        return gb, emu.EmuSearch(gb, rotation_flip=0, **opts)

    (gb0, m0), (gb1, m1) = make(), make()
    for _ in range(3):
        r0 = m0.act(fake_actor(m0, n))
        m1.begin_move()
        for _ in range(m1.waves_per_move):
            assert m1.select(wait=False).shape[0] == m1.max_leaves
            k = m1.leaf_count()
            h = m1.leaf_info()[0]
            assert len(h) == k
            if k == 0:
                m1.expand_backup(None, None)
                continue
            pi, v = oracles.fakenet(h, n * n + 1)
            with pytest.raises(AssertionError):  # fewer rows than the known count
                m1.expand_backup(torch.from_numpy(pi[: k - 1]), torch.from_numpy(v[: k - 1]))
            m1.expand_backup(torch.from_numpy(pi), torch.from_numpy(v))
        r1 = m1.results()
        for key in ("visits", "best_action", "total_visits", "root_value", "best_q"):
            np.testing.assert_array_equal(r0[key], r1[key])
        np.testing.assert_array_equal(m0.root_priors(), m1.root_priors())
        a = r0["best_action"]
        for gb, m in ((gb0, m0), (gb1, m1)):
            assert gb.forward(a).all()
            m.advance(a)
    assert m1.eval_count() == m0.eval_count() and (m1.errors() == 0).all()


def test_bench_search_twin_on_the_kernels(emu):
    """small-G twin of tests/test_gpu_search_at_scale.py on the emulated kernels: 19x19 games with the seeded
    openings of 0..150 plies, binary16 NHWC leaf batches, the asynchronous leaf count, batches padded with NaN
    replies, the plane-reading IntNet (equal probabilities everywhere, std_sort_ties=1), a fresh root and a
    move on the kept tree -- root tables equal the COMPILED reference's, priors bit for bit"""
    from tests import test_gpu_search_at_scale as S

    if not oracles.have_ref(S.N):
        pytest.skip("compiled reference (oracle/_ref) not available")
    G = 4
    opts = dict(S.OPTS, num_rollouts=48)
    games = np.arange(G)
    gb = emu.emu_batch(G, S.N)
    S.play_openings(gb, 0)
    legal = gb.legal_mask()[:, :-1].sum(1)
    assert legal.min() < 256 < legal.max(), legal  # both sort networks of k_expand
    net = S.net()
    want = S.reference_records(games, net, opts)
    mc = emu.EmuSearch(gb, rotation_flip=0, feature_format="f16", cpad=24, std_sort_ties=1, **opts)
    actor = S.PaddedActor(net, [mc], batchsize=12)
    dup = 0
    for move in range(S.MOVES):
        S.async_wave_search(mc, actor)
        res = mc.results()
        dup += S.compare_sample(res, mc.root_priors(), games, want, move)
        assert gb.forward(res["best_action"]).all()
        mc.advance(res["best_action"])
    assert (mc.errors() == 0).all(), mc.errors()
    assert actor.padded > 0 and dup >= G
