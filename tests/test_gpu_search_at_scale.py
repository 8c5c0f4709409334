"""The search configuration bench.py times, on the device, against the reference search.

bench.py searches 4096 19x19 games with 800 rollouts in waves of 8 (virtual loss 1, persistent tree,
c_puct 1.5) as two parts interleaved by WavePipeline, binary16 NHWC leaf batches padded to a multiple of
the network's batch size.  Here that path runs with IntNet (tests/oracles.py: reads the planes, same bits
on device and host, equal probabilities in nearly every reply as an fp16 head, hence std_sort_ties=1), from
seeded openings of 0..150 plies (both sort networks of k_expand), for a fresh root and a kept tree.
A sample of 64 games must reproduce the compiled reference search's root tables: most-visited move, total
visits and root value, plus a digest of every edge's visits and float32 prior
(tests/golden/mcts_19_scale_sample.json, scripts/gen_golden.py; a few are re-searched live when oracle/_ref
is built).  Padded rows are answered with NaN, so reading one cannot go unnoticed.  rotation_flip is off:
the device's D4 stream is not the reference's."""
import hashlib
import json
import os
import time

import numpy as np
import pytest

from tests import oracles

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mcts_19_scale_sample.json")
N, R, B = 19, 800, 8
OPTS = dict(num_rollouts=R, num_rollouts_per_batch=B, virtual_loss=1, persistent_tree=1, c_puct=1.5)
# NN batch 384, not bench.py's 256: 2048 games x 8 leaves fill 256-row batches exactly, nothing would be padded
SEED, MAX_OPEN, SAMPLE, MOVES, NN_BATCH, LIVE = 2026, 150, 64, 2, 384, 4


def net():
    return oracles.int_net(N, levels=24, seed=SEED)


def opening_plan(games):
    """per game, from a generator of its own: opening length (0..MAX_OPEN) and one uniform per ply"""
    rs = [np.random.default_rng([SEED, int(g)]) for g in games]
    return np.array([r.integers(0, MAX_OPEN + 1) for r in rs]), np.array([r.random(MAX_OPEN) for r in rs])


def pick(legal, u):
    """the legal board point at quantile u of each row of legal [k, N*N]"""
    legal = np.asarray(legal, np.int64)
    k = np.minimum((u * legal.sum(1)).astype(np.int64), legal.sum(1) - 1)
    return (np.cumsum(legal, 1) > k[:, None]).argmax(1).astype(np.int32)


def play_openings(gb, first_game):
    lens, u = opening_plan(range(first_game, first_game + gb.num_games))
    for t in range(int(lens.max())):
        acts = pick(gb.legal_mask()[:, :-1], u[:, t])
        acts[lens <= t] = -1
        assert gb.forward(acts)[acts >= 0].all()


def sample_games(G):
    """32 of the first 512 games (the smaller variant) and 32 of the rest of the 4096"""
    rng = np.random.default_rng(SEED)
    g = np.sort(np.concatenate([rng.choice(512, SAMPLE // 2, replace=False),
                                512 + rng.choice(3584, SAMPLE // 2, replace=False)]))
    return g[g < G]


def record(visits, prior, best, total, value):
    """[best action, total visits, root value, digest of the visits of every action (-1 = no edge) and the
    float32 priors of the edges]"""
    v = np.asarray(visits, "<i4")
    p = np.where(v >= 0, prior, -1).astype("<f4")
    return [int(best), int(total), float(np.float32(value)), hashlib.sha256(v.tobytes() + p.tobytes()).hexdigest()[:20]]


def reference_records(games, network=None, opts=OPTS):
    """the compiled reference search's records of `games` ([game][move]), moves on its own choice"""
    network, out = network or net(), []
    for g in games:
        lens, u = opening_plan([g])
        st, rm = oracles.Ref(N), oracles.RefMcts(N, callback=network, **opts)
        for t in range(int(lens[0])):
            assert st.forward(int(pick(st.legal()[None], u[:1, t])[0]))
        out.append([])
        for _ in range(MOVES):
            r = rm.act(st)
            out[-1].append(record(r["visits"], r["prior"], r["best_action"], r["total_visits"], r["root_value"]))
            assert st.forward(r["best_action"])
    return out


class PaddedActor:
    """IntNet on batches padded to `batchsize` rows; the replies of the padded rows are NaN"""

    def __init__(self, network, searches, batchsize=NN_BATCH):
        self.net, self.searches, self.batchsize, self.padded = network, searches, batchsize, 0

    def reply(self, s, n):
        pi, v = self.net.torch(s)
        pi[n:], v[n:] = float("nan"), float("nan")
        self.padded += s.shape[0] - n
        return {"pi": pi, "V": v}

    def __call__(self, batch):  # WavePipeline: the part is found by its feature tensor
        s = batch["s_nhwc"]
        mc = next(m for m in self.searches if s.data_ptr() == m.feat.data_ptr())
        assert 0 < mc._n <= s.shape[0] and (s.shape[0] % self.batchsize == 0 or s.shape[0] == mc.max_leaves)
        return self.reply(s, mc._n)


def async_wave_search(mc, actor):
    """one move, the leaf count fetched after the descents: select(wait=False) -> leaf_count() ->
    leaf_info() -> network on the padded rows -> expand_backup"""
    import torch

    mc.begin_move()
    for _ in range(mc.waves_per_move):
        s = mc.select(wait=False)
        n = mc.leaf_count()
        h, gi, _ = mc.leaf_info()
        assert s.shape[0] == mc.max_leaves and len(h) == len(gi) == n
        assert ((0 <= gi) & (gi < mc.gb.num_games)).all()
        if n == 0:
            mc.expand_backup(None, None)
            continue
        rep = actor.reply(s[:min(-(-n // actor.batchsize) * actor.batchsize, mc.max_leaves)], n)
        if s.is_cuda:  # the reply comes from torch's stream, the expansion runs on the context stream
            torch.cuda.synchronize()
        mc.expand_backup(rep["pi"], rep["V"])


def compare_sample(res, priors, games, want, move):
    """the device's root tables of `games` against the reference's records; returns how many of them have
    bit-equal priors on two root edges"""
    dup = 0
    for i, g in enumerate(games):
        got = record(res["visits"][g], priors[g], res["best_action"][g], res["total_visits"][g], res["root_value"][g])
        assert got[:3] == want[i][move][:3], (g, move, got, want[i][move])
        assert got[3] == want[i][move][3], f"root visits or priors differ: game {g} move {move}"
        p = priors[g][priors[g] >= 0]
        dup += len(np.unique(p)) < len(p)
    return dup


def run_at_scale(G, parts, feature_format, cpad, pipelined):
    import torch

    import elf_b200
    from elf_b200.pipeline import WavePipeline

    free, total = torch.cuda.mem_get_info(0)
    need = 16 * G * 2**20  # the default node pool: about 56 GB at 4096 games (as in bench.py), plus the net
    if free < need:
        pytest.skip(f"needs ~{need / 2**30:.0f} GiB free on the device: "
                    f"{free / 2**30:.0f} of {total / 2**30:.0f} GiB are")
    Gp = G // parts
    gbs = [elf_b200.GoBatch(Gp, board_size=N, device=0) for _ in range(parts)]
    searches = []
    try:
        for p, gb in enumerate(gbs):
            play_openings(gb, p * Gp)
        searches = [elf_b200.MctsBatch(gb, rotation_flip=0, feature_format=feature_format, cpad=cpad, std_sort_ties=1,
                                       **OPTS) for gb in gbs]
        search_gib = (free - torch.cuda.mem_get_info(0)[0]) / 2**30
        stored = json.load(open(GOLD))
        assert stored["opts"] == OPTS and stored["seed"] == SEED
        games = sample_games(G)
        want = [stored["tables"][stored["games"].index(int(g))] for g in games]
        if oracles.have_ref(N):  # the host search takes about a second per game: re-derive a few stored records
            assert reference_records(games[:LIVE]) == want[:LIVE]
        actor = PaddedActor(net(), searches)
        dup, t0 = 0, time.perf_counter()
        for move in range(MOVES):
            if pipelined:
                WavePipeline(searches, actor).search()
            else:
                for mc in searches:
                    async_wave_search(mc, actor)
            torch.cuda.synchronize()
            rs = [mc.results() for mc in searches]
            res = {k: np.concatenate([r[k] for r in rs]) for k in rs[0]}
            for mc in searches:
                assert (mc.errors() == 0).all(), mc.errors()
            assert (res["total_visits"] == R - B).all() if move == 0 else (res["total_visits"] >= R - B).all()
            dup += compare_sample(res, np.concatenate([mc.root_priors() for mc in searches]), games, want, move)
            for p, (gb, mc) in enumerate(zip(gbs, searches)):
                a = np.ascontiguousarray(res["best_action"][p * Gp:(p + 1) * Gp])
                assert gb.forward(a).all()
                mc.advance(a)
        print(f"G={G} {feature_format}/cpad {cpad}: {MOVES * len(games)} root tables equal the reference's, {dup} with "
              f"equal priors; {time.perf_counter() - t0:.1f} s on the device, {actor.padded} padded rows, search state "
              f"{search_gib:.1f} GiB, torch peak {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
        assert actor.padded > 0 and dup >= MOVES * len(games) // 2, (actor.padded, dup)
    finally:  # a failed check must not leave the node pools allocated for the tests after it
        for x in searches + gbs:
            x.close()


@pytest.mark.parametrize("n", [9, 19])
def test_int_net_same_bits_on_device_and_host(n):
    """IntNet on the device (float32 NCHW and 16-bit NHWC planes, several batch shapes, TF32 on and off)
    answers the same bits as its numpy twin"""
    import torch

    network, rng, tf32 = oracles.int_net(n, seed=SEED), np.random.default_rng(n), torch.backends.cuda.matmul.allow_tf32
    try:
        for m in (1, 7, 256, 1000):
            x = (rng.random((m, 18, n, n)) < rng.uniform(0.05, 0.6)).astype(np.float32)
            want = [torch.from_numpy(a).cuda() for a in network.numpy(x)]
            for allow in (False, True):
                torch.backends.cuda.matmul.allow_tf32 = allow
                for dt, cpad in ((None, 0), (torch.float16, 24), (torch.bfloat16, 32)):
                    s = torch.from_numpy(x).cuda()
                    if dt is not None:
                        s = torch.nn.functional.pad(s.permute(0, 2, 3, 1), (0, cpad - 18)).to(dt).contiguous()
                    pi, v = network.torch(s)
                    assert torch.equal(pi, want[0]) and torch.equal(v, want[1]), (m, allow, dt)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32


def test_bench_search_at_4096_games_matches_reference():
    """bench.py's configuration: 4096 games, two parts of 2048 in WavePipeline, f16 NHWC with cpad 24"""
    run_at_scale(4096, 2, "f16", 24, pipelined=True)


def test_bf16_async_count_at_512_games_matches_reference():
    """bf16 NHWC with cpad 32 and the asynchronous leaf count (select(wait=False), leaf_count, leaf_info)"""
    run_at_scale(512, 1, "bf16", 32, pipelined=False)
