"""ctypes wrappers around the TEST-ONLY checkers in oracle/:

* ``Oracle``  -- the C restatement (oracle/go_oracle.c -> oracle/libgo_oracle.so), runtime board size.
* ``Ref``     -- the compiled unmodified reference (oracle/_ref/libref_go{19,9}.so), when present.

Both expose the same methods so tests can be parametrised over them.
"""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
vp = ctypes.c_void_p


def load_oracle():
    path = os.path.join(ORACLE_DIR, "libgo_oracle.so")
    if not os.path.exists(path):
        subprocess.check_call([os.environ.get("PYTHON", "python"), os.path.join(ROOT, "scripts", "gen_zobrist.py")])
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"])
    L = ctypes.CDLL(path)
    L.go_new.restype = vp
    L.go_new.argtypes = [ctypes.c_int]
    L.go_clone.restype = vp
    L.go_clone.argtypes = [vp]
    L.go_free.argtypes = [vp]
    L.go_reset.argtypes = [vp]
    L.go_forward.argtypes = [vp, ctypes.c_int]
    L.go_check_move.argtypes = [vp, ctypes.c_int]
    L.go_hash.restype = ctypes.c_uint64
    L.go_hash.argtypes = [vp]
    L.go_info.argtypes = [vp, vp]
    L.go_stones.argtypes = [vp, vp]
    L.go_legal_mask.argtypes = [vp, vp]
    L.go_true_eye_mask.argtypes = [vp, ctypes.c_int, vp]
    L.go_tt_score.argtypes = [vp]
    L.go_evaluate.restype = ctypes.c_float
    L.go_evaluate.argtypes = [vp, ctypes.c_float]
    L.go_features_agz.argtypes = [vp, ctypes.c_int, vp]
    L.go_d4_action2action.argtypes = [ctypes.c_int] * 3
    L.go_terminated.argtypes = [vp]
    L.go_playout.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int] + [vp] * 5
    L.go_playout_many.restype = ctypes.c_int64
    L.go_playout_many.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    return L


def ref_path(n):
    return os.path.join(ORACLE_DIR, "_ref", f"libref_go{n}.so")


def have_ref(n):
    return os.path.exists(ref_path(n))


_ref_cache = {}


def load_ref(n):
    if n in _ref_cache:
        return _ref_cache[n]
    L = ctypes.CDLL(ref_path(n))
    L.ref_new.restype = vp
    L.ref_clone.restype = vp
    L.ref_clone.argtypes = [vp]
    L.ref_free.argtypes = [vp]
    L.ref_reset.argtypes = [vp]
    L.ref_forward.argtypes = [vp, ctypes.c_int]
    L.ref_hash.restype = ctypes.c_uint64
    L.ref_hash.argtypes = [vp]
    L.ref_info.argtypes = [vp, vp]
    L.ref_stones.argtypes = [vp, vp]
    L.ref_legal_mask.argtypes = [vp, vp]
    L.ref_find_all_valid_moves.argtypes = [vp, vp]
    L.ref_true_eye_mask.argtypes = [vp, ctypes.c_int, vp]
    L.ref_tt_score.argtypes = [vp]
    L.ref_evaluate.restype = ctypes.c_float
    L.ref_evaluate.argtypes = [vp, ctypes.c_float]
    L.ref_features_agz.argtypes = [vp, ctypes.c_int, vp]
    L.ref_d4_action2action.argtypes = [ctypes.c_int] * 2
    L.ref_playout.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int] + [vp] * 5
    assert L.ref_board_size() == n
    _ref_cache[n] = L
    return L


class _Base:
    """One game state with the GoState-like observer set used by the tests."""


class Oracle(_Base):
    def __init__(self, n=19, lib=None):
        self.L = lib or load_oracle()
        self.n = n
        self.p = self.L.go_new(n)

    def __del__(self):
        if getattr(self, "p", None):
            self.L.go_free(self.p)
            self.p = None

    def forward(self, a):
        return bool(self.L.go_forward(self.p, int(a)))

    def hash(self):
        return int(self.L.go_hash(self.p))

    def info(self):
        o = np.zeros(12, np.int32)
        self.L.go_info(self.p, o.ctypes.data)
        return o

    def stones(self):
        o = np.zeros(self.n * self.n, np.uint8)
        self.L.go_stones(self.p, o.ctypes.data)
        return o

    def legal(self):
        o = np.zeros(self.n * self.n, np.uint8)
        self.L.go_legal_mask(self.p, o.ctypes.data)
        return o

    def true_eyes(self, player):
        o = np.zeros(self.n * self.n, np.uint8)
        self.L.go_true_eye_mask(self.p, player, o.ctypes.data)
        return o

    def tt_score(self):
        return int(self.L.go_tt_score(self.p))

    def evaluate(self, komi):
        return float(self.L.go_evaluate(self.p, komi))

    def features(self, d4=0):
        o = np.zeros((18, self.n, self.n), np.float32)
        self.L.go_features_agz(self.p, d4, o.ctypes.data)
        return o

    def terminated(self):
        return bool(self.L.go_terminated(self.p))


def ref_sgf_parse(text, n, cap=2048):
    """the reference's own Sgf::load + main-line iteration (oracle/ref_shim.cc: ref_sgf_parse).
    Returns None if the reference refuses the text, else a dict."""
    L = load_ref(n)
    L.ref_sgf_parse.restype = ctypes.c_int
    L.ref_sgf_parse.argtypes = [ctypes.c_char_p, vp, vp, ctypes.c_int, vp, vp]
    acts = np.zeros(cap, np.int32)
    pl = np.zeros(cap, np.int32)
    hi = np.zeros(4, np.int32)
    hf = np.zeros(2, np.float32)
    k = L.ref_sgf_parse(text.encode("latin-1", "replace"), acts.ctypes.data, pl.ctypes.data, cap, hi.ctypes.data,
                        hf.ctypes.data)
    if k < 0:
        return None
    return {"actions": acts[:k].tolist(), "players": pl[:k].tolist(), "size": int(hi[0]), "handi": int(hi[1]),
            "winner": int(hi[2]), "num_moves": int(hi[3]), "komi": float(hf[0]), "win_margin": float(hf[1])}


def ref_record_roundtrip(text, n=9):
    """Record::createFromJson + setJsonFields of the compiled reference; None if its parser throws"""
    L = load_ref(n)
    L.ref_record_roundtrip.restype = ctypes.c_int
    L.ref_record_roundtrip.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    cap = 4 * len(text) + (1 << 16)
    buf = ctypes.create_string_buffer(cap)
    k = L.ref_record_roundtrip(text.encode(), buf, cap)
    assert k != -2
    return None if k < 0 else buf.value.decode()


def ref_request_roundtrip(text, n=9):
    """MsgRequest::createFromJson + setJsonFields of the compiled reference; None if it throws"""
    L = load_ref(n)
    L.ref_request_roundtrip.restype = ctypes.c_int
    L.ref_request_roundtrip.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    buf = ctypes.create_string_buffer(1 << 16)
    k = L.ref_request_roundtrip(text.encode(), buf, 1 << 16)
    return None if k < 0 else buf.value.decode()


def ref_record_batch_count(text, n=9):
    L = load_ref(n)
    L.ref_record_batch_count.restype = ctypes.c_int
    L.ref_record_batch_count.argtypes = [ctypes.c_char_p]
    return int(L.ref_record_batch_count(text.encode()))


def ref_quantise_policy(actions, visits, n):
    L = load_ref(n)
    L.ref_quantise_policy.restype = ctypes.c_int
    L.ref_quantise_policy.argtypes = [ctypes.c_int, vp, vp, vp]
    a = np.ascontiguousarray(actions, np.int32)
    v = np.ascontiguousarray(visits, np.float32)
    out = np.zeros((n + 2) * (n + 2), np.uint8)
    k = L.ref_quantise_policy(len(a), a.ctypes.data, v.ctypes.data, out.ctypes.data)
    assert k == out.size
    return out


def ref_should_resign(resign_thres, never_resign, value, next_player, ply, n=9):
    """the reference's ResignCheck::check through GoStateExt::shouldResign's colour handling and the
    ply >= 50 test of GoGameSelfPlay::act (oracle/ref_offline_shim.cc)"""
    L = load_ref(n)
    L.ref_should_resign.restype = ctypes.c_int
    L.ref_should_resign.argtypes = [ctypes.c_float, ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int]
    return bool(L.ref_should_resign(float(resign_thres), int(never_resign), float(value), int(next_player), int(ply)))


def ref_offline_sample(record_json, move_to, d4, num_future, n):
    """one training sample from the reference's GoStateExtOffline + GoFeature extractors"""
    L = load_ref(n)
    L.ref_offline_sample.restype = ctypes.c_int
    L.ref_offline_sample.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, vp, vp]
    s = np.zeros((18, n, n), np.float32)
    oa = np.zeros(num_future, np.int64)
    sc = np.zeros(n * n + 1, np.float32)
    fl = np.zeros(2, np.float32)
    it = np.zeros(3, np.int32)
    ver = np.zeros(1, np.int64)
    rc = L.ref_offline_sample(record_json.encode(), int(move_to), int(d4), int(num_future), s.ctypes.data, oa.ctypes.data,
                              sc.ctypes.data, fl.ctypes.data, it.ctypes.data, ver.ctypes.data)
    if rc != 0:
        return rc
    return {"s": s, "offline_a": oa, "mcts_scores": sc, "winner": float(fl[0]), "predicted_value": float(fl[1]),
            "move_idx": int(it[0]), "num_move": int(it[1]), "aug_code": int(it[2]), "selfplay_ver": int(ver[0])}


def ref_show_board(ref):
    L = ref.L
    L.ref_show_board.restype = ctypes.c_int
    L.ref_show_board.argtypes = [vp, ctypes.c_char_p, ctypes.c_int]
    buf = ctypes.create_string_buffer(4096)
    k = L.ref_show_board(ref.p, buf, 4096)
    assert k >= 0
    return buf.value.decode()


def ref_vertex_str(n, action):
    L = load_ref(n)
    L.ref_vertex_str.restype = ctypes.c_int
    L.ref_vertex_str.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    buf = ctypes.create_string_buffer(32)
    assert L.ref_vertex_str(int(action), buf, 32) >= 0
    return buf.value.decode()


class Ref(_Base):
    def __init__(self, n=19):
        self.L = load_ref(n)
        self.n = n
        self.p = self.L.ref_new()

    def __del__(self):
        if getattr(self, "p", None):
            self.L.ref_free(self.p)
            self.p = None

    def forward(self, a):
        return bool(self.L.ref_forward(self.p, int(a)))

    def hash(self):
        return int(self.L.ref_hash(self.p))

    def info(self):
        o = np.zeros(12, np.int32)
        self.L.ref_info(self.p, o.ctypes.data)
        return o

    def stones(self):
        o = np.zeros(self.n * self.n, np.uint8)
        self.L.ref_stones(self.p, o.ctypes.data)
        return o

    def legal(self):
        o = np.zeros(self.n * self.n, np.uint8)
        self.L.ref_legal_mask(self.p, o.ctypes.data)
        return o

    def true_eyes(self, player):
        o = np.zeros(self.n * self.n, np.uint8)
        self.L.ref_true_eye_mask(self.p, player, o.ctypes.data)
        return o

    def tt_score(self):
        return int(self.L.ref_tt_score(self.p))

    def evaluate(self, komi):
        return float(self.L.ref_evaluate(self.p, komi))

    def features(self, d4=0):
        o = np.zeros((18, self.n, self.n), np.float32)
        self.L.ref_features_agz(self.p, d4, o.ctypes.data)
        return o

    def terminated(self):
        return bool(self.info()[9])

    def features_df(self, d4=0):
        """BoardFeature::extract: the 25 DarkForest planes"""
        o = np.zeros((25, self.n, self.n), np.float32)
        self.L.ref_features_df.argtypes = [vp, ctypes.c_int, vp]
        self.L.ref_features_df.restype = None
        self.L.ref_features_df(self.p, int(d4), o.ctypes.data)
        return o


def oracle_playout(n, seed, gid, max_plies=None, trace=False, lib=None):
    L = lib or load_oracle()
    max_plies = max_plies or 2 * n * n
    chk = ctypes.c_uint64()
    sc = ctypes.c_int32()
    if trace:
        moves = np.zeros(max_plies, np.int32)
        hashes = np.zeros(max_plies, np.uint64)
        caps = np.zeros(2 * max_plies, np.int32)
        t = L.go_playout(n, seed, gid, max_plies, moves.ctypes.data, hashes.ctypes.data, caps.ctypes.data,
                         ctypes.byref(chk), ctypes.byref(sc))
        return t, chk.value, sc.value, moves[:t], hashes[:t], caps[: 2 * t].reshape(-1, 2)
    t = L.go_playout(n, seed, gid, max_plies, None, None, None, ctypes.byref(chk), ctypes.byref(sc))
    return t, chk.value, sc.value


def oracle_playout_many(n, seed, first, count, max_plies=None, lib=None):
    L = lib or load_oracle()
    max_plies = max_plies or 2 * n * n
    chk = np.zeros(count, np.uint64)
    plies = np.zeros(count, np.int32)
    score = np.zeros(count, np.int32)
    tot = L.go_playout_many(n, seed, first, count, max_plies, chk.ctypes.data, plies.ctypes.data, score.ctypes.data)
    return {"chk": chk, "plies": plies, "score": score, "total_plies": int(tot)}


def ref_playout(n, seed, gid, max_plies=None):
    L = load_ref(n)
    max_plies = max_plies or 2 * n * n
    chk = ctypes.c_uint64()
    sc = ctypes.c_int32()
    t = L.ref_playout(seed, gid, max_plies, None, None, None, ctypes.byref(chk), ctypes.byref(sc))
    return t, chk.value, sc.value


# group accessors (reference Board::_groups) -------------------------------------------------
def _bind_groups():
    L = load_oracle()
    for f in ("go_group_liberties", "go_group_stones"):
        getattr(L, f).argtypes = [vp, ctypes.c_int]
    L.go_num_groups.argtypes = [vp]


def oracle_group(o, action):
    _bind_groups()
    return int(o.L.go_group_liberties(o.p, action)), int(o.L.go_group_stones(o.p, action))


def oracle_num_groups(o):
    _bind_groups()
    return int(o.L.go_num_groups(o.p))


def ref_group(r, action):
    r.L.ref_group_liberties.argtypes = [vp, ctypes.c_int]
    r.L.ref_group_stones.argtypes = [vp, ctypes.c_int]
    return int(r.L.ref_group_liberties(r.p, action)), int(r.L.ref_group_stones(r.p, action))


def ref_num_groups(r):
    r.L.ref_num_groups.argtypes = [vp]
    return int(r.L.ref_num_groups(r.p))


# ---- deterministic fake network (oracle/fakenet.h) in numpy -------------------------------
_GOLD = np.uint64(0x9E3779B97F4A7C15)


def _splitmix64(x):
    with np.errstate(over="ignore"):
        x = x + _GOLD
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))


def fakenet(hashes, num_actions):
    """bit-exact numpy twin of oracle/fakenet.h: returns (pi float32 [n, A], v float32 [n])"""
    h = np.asarray(hashes, dtype=np.uint64).reshape(-1, 1)
    a = (np.arange(num_actions, dtype=np.uint64) + np.uint64(1)).reshape(1, -1)
    with np.errstate(over="ignore"):
        r = _splitmix64(h ^ (a * _GOLD))
    u = ((r >> np.uint64(40)) + np.uint64(1)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    t = u * u
    t = t * t
    t = t * t
    r2 = _splitmix64(h[:, 0] ^ np.uint64(0x5EED5EED))
    v = (r2 >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 8388608.0) - np.float32(1.0)
    return t.astype(np.float32), v.astype(np.float32)


class RefMcts:
    """the reference search (MCTSAI_T + MCTSActor logic) through oracle/_ref, fake net or callback"""

    def __init__(self, n, num_rollouts=200, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1,
                 use_prior=1, unexplored_q_zero=0, root_unexplored_q_zero=0, ply_pass_enabled=0,
                 remove_pass_if_dangerous=1, seed=7, c_puct=1.5, komi=7.5, callback=None, root_epsilon=0.0,
                 root_alpha=0.0, rotation_flip=0):
        self.L = load_ref(n)
        self.n = n
        L = self.L
        L.ref_mcts_new.restype = vp
        L.ref_mcts_new.argtypes = [vp, vp, vp]
        L.ref_mcts_act.argtypes = [vp, vp] + [vp] * 6
        L.ref_mcts_free.argtypes = [vp]
        L.ref_mcts_num_evals.restype = ctypes.c_long
        L.ref_mcts_num_evals.argtypes = [vp]
        iopts = np.array([num_rollouts, num_rollouts_per_batch, virtual_loss, persistent_tree, use_prior,
                          unexplored_q_zero, root_unexplored_q_zero, ply_pass_enabled, remove_pass_if_dangerous,
                          int(seed) & 0x7FFFFFFF, 1], np.int32)  # [9] only feeds TSOptions::seed (unused by the search)
        fopts = np.array([c_puct, komi, root_epsilon, root_alpha], np.float32)
        self._cb = None
        if callback is not None:
            CB = ctypes.CFUNCTYPE(None, ctypes.c_int, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint64),
                                  ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float))
            P1 = n * n + 1

            def tramp(cnt, feats, hashes, pi, v):
                f = np.ctypeslib.as_array(feats, shape=(cnt, 18, n, n))
                h = np.ctypeslib.as_array(hashes, shape=(cnt,))
                p, val = callback(f, h)
                np.ctypeslib.as_array(pi, shape=(cnt, P1))[:] = p
                np.ctypeslib.as_array(v, shape=(cnt,))[:] = val

            self._cb = CB(tramp)
        L.ref_mcts_new_ex.restype = vp
        L.ref_mcts_new_ex.argtypes = [vp, vp, vp, ctypes.c_int, ctypes.c_uint32]
        L.ref_mcts_last_order.argtypes = [vp, vp]
        L.ref_mcts_sample.argtypes = [vp, vp]
        cbp = ctypes.cast(self._cb, vp) if self._cb else None
        # seed: MCTSActorParams::seed, a full 32-bit value when it comes from the game thread's generator
        self.m = L.ref_mcts_new_ex(iopts.ctypes.data, fopts.ctypes.data, cbp, int(rotation_flip), int(seed) & 0xFFFFFFFF)

    def end_game(self, ref_state):
        """MCTSAI_T::endGame: the tree is reset (finish_game, game_selfplay.cc:139-143)"""
        self.L.ref_mcts_end_game.argtypes = [vp, vp]
        self.L.ref_mcts_end_game(self.m, ref_state.p)

    def last_order(self):
        """actions of the root edges in the order MCTSResultT::addActions walked the container"""
        a = np.zeros(self.n * self.n + 1, np.int32)
        k = self.L.ref_mcts_last_order(self.m, a.ctypes.data)
        return a[:k].copy()

    def sample(self, rng):
        """mcts_make_diverse_move's sampling on the game thread's generator (a RefRng)"""
        return int(self.L.ref_mcts_sample(self.m, rng.p))

    def act(self, ref_state, policy_only=False):
        """MCTSAI_T::act, or actPolicyOnly (the move of a *_use_policy_network_only colour)"""
        P1 = self.n * self.n + 1
        vis = np.zeros(P1, np.int32)
        w = np.zeros(P1, np.float32)
        pr = np.zeros(P1, np.float32)
        rv = ctypes.c_float()
        bq = ctypes.c_float()
        tv = ctypes.c_int32()
        fn = self.L.ref_mcts_act_policy_only if policy_only else self.L.ref_mcts_act
        fn.argtypes = [vp, vp] + [vp] * 6
        a = fn(self.m, ref_state.p, vis.ctypes.data, w.ctypes.data, pr.ctypes.data,
               ctypes.byref(rv), ctypes.byref(bq), ctypes.byref(tv))
        return {"best_action": int(a), "visits": vis, "wsum": w, "prior": pr, "root_value": rv.value,
                "best_q": bq.value, "total_visits": tv.value}

    def num_evals(self):
        return int(self.L.ref_mcts_num_evals(self.m))

    def __del__(self):
        if getattr(self, "m", None):
            self.L.ref_mcts_free(self.m)
            self.m = None


class RefRng:
    """a reference game thread's std::mt19937 (GoGameBase::_rng) through oracle/_ref"""

    def __init__(self, n, seed):
        self.L = L = load_ref(n)
        L.ref_rng_new.restype = vp
        L.ref_rng_new.argtypes = [ctypes.c_uint64]
        L.ref_rng_free.argtypes = [vp]
        L.ref_rng_next.restype = ctypes.c_uint32
        L.ref_rng_next.argtypes = [vp]
        self.p = L.ref_rng_new(int(seed))

    def next(self):
        return int(self.L.ref_rng_next(self.p))

    def __del__(self):
        if getattr(self, "p", None):
            self.L.ref_rng_free(self.p)
            self.p = None


class RefResign:
    """the reference's ResignCheck as GoStateExt::shouldResign drives it, with its random draw"""

    def __init__(self, n, thres, never_resign_ratio):
        self.L = L = load_ref(n)
        L.ref_resign_new.restype = vp
        L.ref_resign_new.argtypes = [ctypes.c_float, ctypes.c_float]
        L.ref_resign_free.argtypes = [vp]
        L.ref_resign_reset.argtypes = [vp]
        L.ref_resign_check.argtypes = [vp, ctypes.c_float, ctypes.c_int, vp]
        self.p = L.ref_resign_new(float(thres), float(never_resign_ratio))

    def check(self, value, next_player, rng):
        return bool(self.L.ref_resign_check(self.p, float(value), int(next_player), rng.p))

    def reset(self):
        self.L.ref_resign_reset(self.p)

    def __del__(self):
        if getattr(self, "p", None):
            self.L.ref_resign_free(self.p)
            self.p = None


class OracleMcts:
    """the C restatement of the search (oracle/mcts_oracle.c); same interface as RefMcts but acts
    on Oracle states"""

    def __init__(self, n, num_rollouts=200, num_rollouts_per_batch=8, virtual_loss=1, persistent_tree=1,
                 use_prior=1, unexplored_q_zero=0, root_unexplored_q_zero=0, ply_pass_enabled=0,
                 remove_pass_if_dangerous=1, seed=7, c_puct=1.5, komi=7.5, lib=None, std_sort_ties=0, callback=None):
        self.L = lib or load_oracle()
        self.n = n
        L = self.L
        L.mo_new.restype = vp
        L.mo_new.argtypes = [ctypes.c_int, vp, vp, vp]
        L.mo_act.argtypes = [vp, vp] + [vp] * 6
        L.mo_free.argtypes = [vp]
        L.mo_num_evals.restype = ctypes.c_long
        L.mo_num_evals.argtypes = [vp]
        iopts = np.array([num_rollouts, num_rollouts_per_batch, virtual_loss, persistent_tree, use_prior,
                          unexplored_q_zero, root_unexplored_q_zero, ply_pass_enabled, remove_pass_if_dangerous,
                          seed, 1, std_sort_ties], np.int32)
        fopts = np.array([c_puct, komi, 0, 0], np.float32)
        self._cb = None
        if callback is not None:  # callback(feats [1,18,n,n], hashes [1]) -> (pi [1,P1], v [1]), as RefMcts
            CB = ctypes.CFUNCTYPE(None, ctypes.c_int, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint64),
                                  ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float))
            P1 = n * n + 1

            def tramp(cnt, feats, hashes, pi, v):
                f = np.ctypeslib.as_array(feats, shape=(cnt, 18, n, n))
                h = np.ctypeslib.as_array(hashes, shape=(cnt,))
                p, val = callback(f, h)
                np.ctypeslib.as_array(pi, shape=(cnt, P1))[:] = p
                np.ctypeslib.as_array(v, shape=(cnt,))[:] = val

            self._cb = CB(tramp)
        self.m = L.mo_new(n, iopts.ctypes.data, fopts.ctypes.data, ctypes.cast(self._cb, vp) if self._cb else None)

    def act(self, oracle_state):
        P1 = self.n * self.n + 1
        vis = np.zeros(P1, np.int32)
        w = np.zeros(P1, np.float32)
        pr = np.zeros(P1, np.float32)
        rv = ctypes.c_float()
        bq = ctypes.c_float()
        tv = ctypes.c_int32()
        a = self.L.mo_act(self.m, oracle_state.p, vis.ctypes.data, w.ctypes.data, pr.ctypes.data,
                          ctypes.byref(rv), ctypes.byref(bq), ctypes.byref(tv))
        return {"best_action": int(a), "visits": vis, "wsum": w, "prior": pr, "root_value": rv.value,
                "best_q": bq.value, "total_visits": tv.value}

    def num_evals(self):
        return int(self.L.mo_num_evals(self.m))

    def last_order(self):
        """actions of the root edges in the reference's container order (as RefMcts.last_order)"""
        a = np.zeros(self.n * self.n + 1, np.int32)
        self.L.mo_last_order.argtypes = [vp, vp]
        k = self.L.mo_last_order(self.m, a.ctypes.data)
        return a[:k].copy()

    def prefix_stats(self):
        """(violations, checks) of the selected-prefix property the CUDA select kernel relies on"""
        self.L.mo_prefix_violations.restype = ctypes.c_long
        self.L.mo_prefix_violations.argtypes = [vp]
        self.L.mo_prefix_checks.restype = ctypes.c_long
        self.L.mo_prefix_checks.argtypes = [vp]
        return int(self.L.mo_prefix_violations(self.m)), int(self.L.mo_prefix_checks(self.m))

    def tie_stats(self):
        """(descent steps decided by the container-order tie-break, of which beyond the scanned prefix)"""
        for f in (self.L.mo_tie_breaks, self.L.mo_tie_breaks_beyond_prefix):
            f.restype, f.argtypes = ctypes.c_long, [vp]
        return int(self.L.mo_tie_breaks(self.m)), int(self.L.mo_tie_breaks_beyond_prefix(self.m))

    def __del__(self):
        if getattr(self, "m", None):
            self.L.mo_free(self.m)
            self.m = None


def oracle_playout_stream(n, seed, first, slot, num_slots, budget, lib=None):
    L = lib or load_oracle()
    L.go_playout_stream.argtypes = [ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_int, vp, vp]
    acc = ctypes.c_uint64()
    games = ctypes.c_int32()
    t = L.go_playout_stream(n, seed, first, slot, num_slots, budget, ctypes.byref(acc), ctypes.byref(games))
    return t, acc.value, games.value


def feature_net(x, num_actions):
    """deterministic test net computed FROM THE PLANES (not the leaf hash): x float [m,18,N,N] ->
    (pi float32 [m,A], v float32 [m]).  Rows are independent and evaluated in float64 on the CPU, so
    the answer for a position does not depend on the batch it arrives in."""
    x = np.asarray(x, np.float64).reshape(len(x), -1)
    rng = np.random.default_rng(x.shape[1] * 1000003 + num_actions)
    W = rng.standard_normal((x.shape[1], num_actions)) * 0.05
    w2 = rng.standard_normal(x.shape[1]) * 0.02
    z = x @ W
    z -= z.max(1, keepdims=True)
    p = np.exp(z)
    p /= p.sum(1, keepdims=True)
    return p.astype(np.float32), np.tanh(x @ w2).astype(np.float32)


class IntNet:
    """deterministic test net computed FROM THE PLANES whose answer is the same bits on the device
    (torch, any batch shape, any GEMM summation order, TF32 or not) and on the host (numpy).

    logits = planes (0/1) . W with W integer in [-7, 7]: every partial sum is an integer of magnitude
    below 18*361*7 < 2^24, exact in float32 in any order.  pi = TABLE[bucket(logit)] with TABLE[k] =
    2^((k - levels + 1) / 4), left unnormalised like ``fakenet`` (pi2response renormalises over the
    legal moves); few buckets -> bit-equal probabilities among the legal moves of almost every reply, as a
    half-precision network produces them.  v = clamp(planes . w_v, -1023, 1023) / 1024, exact."""

    def __init__(self, n, levels=24, seed=0):
        rng = np.random.default_rng([n, levels, seed])
        K, A = 18 * n * n, n * n + 1
        self.n, self.levels = n, int(levels)
        self.W = rng.integers(-7, 8, size=(K, A)).astype(np.int64)
        self.w_v = rng.integers(-7, 8, size=K).astype(np.int64)
        self.table = np.exp2((np.arange(levels) - (levels - 1)) / 4.0).astype(np.float32)
        # a reply's logits spread with the standard deviation of a sum of ~n*n uniform terms (4.3 n):
        # the middle bucket sits at 0 and `levels` buckets cover about +-2 of those deviations
        self.den = int(np.ceil(4 * 4.3 * n))
        self._dev = {}

    def _bucket(self, logit, floordiv, clip):
        return clip(floordiv(logit * self.levels, self.den) + self.levels // 2, 0, self.levels - 1)

    def numpy(self, x):
        """x: planes [m, 18, n, n] (any dtype holding 0/1) -> (pi float32 [m, A], v float32 [m])"""
        x = np.asarray(x).reshape(len(x), -1)
        assert ((x == 0) | (x == 1)).all()
        if not hasattr(self, "_W64"):  # integer sums far below 2^53: float64 products are exact
            self._W64 = np.concatenate([self.W, self.w_v[:, None]], 1).astype(np.float64)
        z = np.rint(x.astype(np.float64) @ self._W64).astype(np.int64)
        logit, lv = z[:, :-1], z[:, -1]
        pi =self.table[self._bucket(logit, np.floor_divide, np.clip)]
        v = (np.clip(lv, -1023, 1023).astype(np.float32) / np.float32(1024)).astype(np.float32)
        return pi.astype(np.float32), v

    def __call__(self, feats, hashes=None):
        """the RefMcts / OracleMcts callback signature"""
        return self.numpy(feats)

    def torch(self, s):
        """s: CUDA planes, float32 NCHW [m, 18, n, n] or 16-bit NHWC [m, n, n, cpad] (planes in
        channels 0..17) -> (pi float32 [m, A], v float32 [m]) on s's device"""
        import torch

        dev = s.device
        if dev not in self._dev:
            W = torch.from_numpy(np.concatenate([self.W, self.w_v[:, None]], 1).astype(np.float32)).to(dev)
            self._dev[dev] = (W, torch.from_numpy(self.table).to(dev))
        W, table = self._dev[dev]
        x = s.float() if s.dim() == 4 and s.shape[1] == 18 and s.shape[-1] == self.n else s[..., :18].float().permute(0, 3, 1, 2)
        z = torch.round(x.reshape(x.shape[0], -1) @ W).to(torch.int64)
        logit, lv = z[:, :-1], z[:, -1]
        pi = table[self._bucket(logit, lambda a, b: torch.div(a, b, rounding_mode="floor"), torch.clamp)]
        v =torch.clamp(lv, -1023, 1023).to(torch.float32) / 1024
        return pi.contiguous(), v.contiguous()


def int_net(n, levels=24, seed=0):
    """see IntNet"""
    return IntNet(n, levels, seed)
