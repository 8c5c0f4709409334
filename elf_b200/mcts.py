"""MctsBatch: the batched GPU tree search, mirroring the reference's MCTSGoAI for G games at once.

Reference: ``src_cpp/elf/ai/tree_search/mcts.h:29-170`` (MCTSAI_T::act), ``tree_search.h``
(TreeSearchT::run / batch_rollouts), ``src_cpp/elfgames/go/mcts/mcts.h:351-381`` (MCTSGoAI) and
the Python NN callback ``src_py/rlpytorch/trainer/trainer.py:73-115`` (Evaluator.actor), whose
contract is kept: ``actor(batch) -> {"pi": [n, N*N+1], "V": [n]}`` with ``batch["s"]`` a CUDA
float tensor ``[n, 18, N, N]``.
"""
import ctypes

import numpy as np

from . import lib as _l
from .refstream import RefStreamSearch


class MctsBatch(RefStreamSearch):
    """``feature_format``: "f32" = the GoFeature contract, ``batch["s"]`` float32 ``[n,18,N,N]``
    (default); "f16" / "bf16" = the fast mode for a half-precision channels-last network: the leaf
    batch is written as ``batch["s_nhwc"]`` ``[n,N,N,cpad]`` (planes in channels 0..17, zeros above),
    which ``elf_b200.model.FusedActor`` consumes without a cast/permute pass.
    ``std_sort_ties=1`` (a search option like the others, ``include/elfb200_mcts.h``): moves whose network
    probabilities are bit-equal are stored in the order ``std::sort`` leaves them in inside the reference's
    ``pi2response`` instead of by ascending move -- needed to replay the reference's games exactly with a
    half-precision network.
    ``strict_root``: raise when a persistent root does not match the board it is asked to search
    (the reference throws, tree_search.h:488-492); off = count it in ``errors()[0]`` and carry on
    with the tree rebuilt from the board."""

    def __init__(self, go_batch, feature_format="f32", cpad=24, strict_root=True, **opts):
        import torch

        self.gb = go_batch
        self._lib = _l.load_library()
        if feature_format not in ("f32", "f16", "bf16"):
            raise ValueError("feature_format must be f32, f16 or bf16")
        self.feature_format, self.cpad, self.strict_root = feature_format, int(cpad), bool(strict_root)
        self._mismatches = 0
        o = _l.MctsOptions()
        _l.check(self._lib, self._lib.elfb200_mcts_default_options(ctypes.byref(o)))
        for k, v in opts.items():
            if not hasattr(o, k):
                raise TypeError(f"unknown MCTS option {k}")
            setattr(o, k, v)
        self.options = o
        self._m = _l.vp()
        _l.check(self._lib, self._lib.elfb200_mcts_create(go_batch._ctx, ctypes.byref(o), ctypes.byref(self._m)))
        import weakref

        go_batch._children.append(weakref.ref(self))
        n = go_batch.board_size
        self.waves_per_move = self._lib.elfb200_mcts_waves_per_move(self._m)
        self.max_leaves = self._lib.elfb200_mcts_max_leaves(self._m)
        self._torch = torch
        self.device = torch.device("cuda", go_batch.device)
        # the leaf feature batch handed to the network: lives on the device, written in place
        self.set_feature_format(feature_format, cpad)
        self._stream = torch.cuda.ExternalStream(go_batch.stream, device=self.device)
        self._keep = None  # network replies still being read by kernels on the context stream

    def set_feature_format(self, feature_format, cpad=None):
        """switch the leaf-batch format between moves/waves (re-allocates the feature tensor)"""
        torch = self._torch
        if feature_format not in ("f32", "f16", "bf16"):
            raise ValueError("feature_format must be f32, f16 or bf16")
        self.gb.synchronize()
        self.feature_format = feature_format
        self.cpad = self.cpad if cpad is None else int(cpad)
        n = self.gb.board_size
        self.feat = None
        if feature_format == "f32":
            self._fmt = _l.FEAT_F32_NCHW
            self.feat = torch.zeros((self.max_leaves, 18, n, n), dtype=torch.float32, device=self.device)
        else:
            self._fmt = _l.FEAT_F16_NHWC if feature_format == "f16" else _l.FEAT_BF16_NHWC
            dt = torch.float16 if feature_format == "f16" else torch.bfloat16
            self.feat = torch.zeros((self.max_leaves, n, n, self.cpad), dtype=dt, device=self.device)
        self.feat_key = "s" if feature_format == "f32" else "s_nhwc"

    def close(self):
        if getattr(self, "_m", None):
            # the search handle points into the board context: if that is already gone (interpreter
            # shutdown can finalise objects in any order) the handle must not be touched any more
            if getattr(self.gb, "_ctx", None):
                self._lib.elfb200_mcts_destroy(self._m)
            self._m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, mask=None):
        self._ref_settle()
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        _l.check(self._lib, self._lib.elfb200_mcts_reset(self._m, m.ctypes.data if m is not None else None))

    def begin_move(self, active=None):
        self._ref_settle()
        a = None if active is None else np.ascontiguousarray(active, dtype=np.uint8)
        _l.check(self._lib, self._lib.elfb200_mcts_begin_move(self._m, a.ctypes.data if a is not None else None))
        self._ref_begin(a)
        if self.strict_root:
            bad = int(self.errors()[0])
            if bad != self._mismatches:
                n, self._mismatches = bad - self._mismatches, bad
                raise _l.ElfB200Error(
                    f"TreeSearch::Root state is not the same as the input state in {n} game(s): the board moved "
                    "without advance()/reset() of the search (the stale trees were discarded)")

    def select(self, wait=True):
        """one wave of descents; returns the CUDA feature tensor view of the leaves that need the
        network (``[n,18,N,N]`` float32, or ``[n,N,N,cpad]`` in the 16-bit formats; n may be 0).
        ``wait=False``: nothing is read back and the host does not wait -- the view covers all
        ``max_leaves`` rows (rows past the device-side count are stale, their replies are ignored);
        ``leaf_count()`` fetches the count later."""
        n = ctypes.c_int32()
        _l.check(self._lib, self._lib.elfb200_mcts_select_ex(self._m, self.feat.data_ptr(), self._fmt, self.cpad,
                                                             ctypes.byref(n) if wait else None))
        self._n = n.value if wait else -1
        return self.feat[: n.value] if wait else self.feat

    def leaf_features_again(self, out=None, fmt=None, cpad=None):
        """write the planes of the pending leaves once more (default: into the batch tensor, same
        format); asynchronous on the context stream"""
        t = self.feat if out is None else out
        _l.check(self._lib, self._lib.elfb200_mcts_leaf_features(self._m, t.data_ptr(), self._fmt if fmt is None else fmt,
                                                                 self.cpad if cpad is None else cpad))

    def leaf_count(self):
        """the number of leaves of the last wave (waits for the context stream); after
        ``select(wait=False)`` it also becomes the row count ``leaf_info`` / ``expand_backup`` use"""
        n = ctypes.c_int32()
        _l.check(self._lib, self._lib.elfb200_mcts_leaf_count(self._m, ctypes.byref(n)))
        self._n = n.value
        return n.value

    def leaf_info(self):
        n = self._n if self._n >= 0 else self.leaf_count()
        h = np.empty(n, np.uint64)
        g = np.empty(n, np.int32)
        p = np.empty(n, np.int32)
        self.leaf_d4 = np.empty(n, np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_leaf_info(self._m, h.ctypes.data, g.ctypes.data, p.ctypes.data,
                                                             self.leaf_d4.ctypes.data))
        return h, g, p

    def expand_backup(self, pi, v):
        """pi: CUDA float32 [n, N*N+1], v: CUDA float32 [n] (contiguous), produced on any stream
        the caller has synchronised with the context stream."""
        if self._n != 0:
            assert pi.is_cuda and v.is_cuda and pi.dtype == self._torch.float32 and v.dtype == self._torch.float32
            assert pi.is_contiguous() and v.is_contiguous()
            assert pi.shape[0] >= (self._n if self._n > 0 else self.max_leaves)
            _l.check(self._lib, self._lib.elfb200_mcts_expand_backup(self._m, pi.data_ptr(), v.data_ptr()))
            # the kernels read pi / v on the context stream, which the caching allocator knows nothing
            # about: keep the tensors alive until the next wave has been ordered behind them
            self._keep = (pi, v)
        else:
            _l.check(self._lib, self._lib.elfb200_mcts_expand_backup(self._m, None, None))

    def results(self):
        G, P1 = self.gb.num_games, self.gb.num_actions
        best = np.empty(G, np.int32)
        visits = np.empty((G, P1), np.int32)
        rootv = np.empty(G, np.float32)
        bestq = np.empty(G, np.float32)
        tot = np.empty(G, np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_results(
            self._m, best.ctypes.data, visits.ctypes.data, rootv.ctypes.data, bestq.ctypes.data, tot.ctypes.data))
        return {"best_action": best, "visits": visits, "root_value": rootv, "best_q": bestq, "total_visits": tot}

    def choose(self, policy_distri_cutoff, resign_thres, never_resign=None, seed=0):
        """device-side move choice (sample ~ visits while ply <= cutoff, else most visited; -1 =
        resign, -2 = not searched); returns (actions int32[G], values float32[G])"""
        G = self.gb.num_games
        a = np.empty(G, np.int32)
        v = np.empty(G, np.float32)
        nr = None if never_resign is None else np.ascontiguousarray(never_resign, dtype=np.uint8)
        _l.check(self._lib, self._lib.elfb200_mcts_choose(
            self._m, int(policy_distri_cutoff), float(resign_thres), nr.ctypes.data if nr is not None else None,
            int(seed) & 0xFFFFFFFFFFFFFFFF, a.ctypes.data, v.ctypes.data))
        return a, v

    def advance(self, actions):
        self._ref_settle()
        a = np.ascontiguousarray(actions, dtype=np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_advance(self._m, a.ctypes.data))

    def root_priors(self):
        """float32 [G, N*N+1]: prior of every root edge by action, -1 where there is no edge"""
        o = np.empty((self.gb.num_games, self.gb.num_actions), np.float32)
        _l.check(self._lib, self._lib.elfb200_mcts_root_priors(self._m, o.ctypes.data))
        return o

    def errors(self):
        e = np.zeros(4, np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_errors(self._m, e.ctypes.data))
        return e

    def eval_count(self):
        return self._lib.elfb200_mcts_eval_count(self._m)

    def timings(self, reset=False):
        """(ms[4] = select, features, expand, backup kernel time; number of waves)"""
        ms = np.zeros(4, np.float64)
        w = ctypes.c_int64()
        _l.check(self._lib, self._lib.elfb200_mcts_timings(self._m, ms.ctypes.data, ctypes.byref(w), int(reset)))
        return ms, w.value

    def stats(self):
        """uint64[4]: descent steps, edge records read, nodes created, stored edges of visited nodes"""
        s = np.zeros(4, np.uint64)
        _l.check(self._lib, self._lib.elfb200_mcts_stats(self._m, s.ctypes.data))
        return s

    # -- MCTSAI_T::act for all games -----------------------------------------------------------
    def act(self, actor, active=None):
        """Run one full search (all waves) with ``actor(batch) -> {"pi", "V"}`` as the network
        callback and return the root statistics.  The callback sees ``batch["s"]`` on the GPU."""
        self.search(actor, active)
        return self.results()

    def wave(self, actor):
        """one wave: descents, the network on the claimed leaves, expansion and backup.  The host
        waits once (for the leaf count); network and search kernels are ordered by stream events."""
        self.wave_finish(self.wave_eval(actor, self.wave_select()))

    # -- the three pieces of a wave (elf_b200.pipeline.WavePipeline interleaves them across batches) --
    def wave_select(self):
        """descents + leaf features; returns the (padded) feature view for the network or None"""
        pad = int(getattr(self, "_pad", 0) or 0)
        s = self.select()  # waits for the context stream to learn the leaf count
        if s.shape[0] == 0:
            return None
        if pad > 1:
            # static NN shapes: round the batch up to a multiple of the actor's batch size
            # (rows past n are stale features; their replies are never read)
            s = self.feat[: min(-(-s.shape[0] // pad) * pad, self.max_leaves)]
        return s

    def wave_eval(self, actor, s, nn_stream=None):
        """enqueue the network on ``nn_stream`` (default: torch's current stream) behind the feature
        kernel; returns (pi, v, event) or None"""
        if s is None:
            return None
        torch = self._torch
        st = nn_stream if nn_stream is not None else torch.cuda.current_stream(self.device)
        st.wait_stream(self._stream)  # the network after the features
        with torch.cuda.stream(st), torch.no_grad():
            reply = actor({self.feat_key: s})
            pi = reply["pi"].to(torch.float32).contiguous()
            v = reply["V"].to(torch.float32).reshape(-1).contiguous()
            ev = torch.cuda.Event()
            ev.record(st)
        return pi, v, ev

    def wave_finish(self, reply):
        """expansion + backup on the context stream, behind the network's event; does not wait"""
        if reply is None:
            self.expand_backup(None, None)
            return
        pi, v, ev = reply
        self._stream.wait_event(ev)
        self.expand_backup(pi, v)

    def search(self, actor, active=None, waves=None):
        """the search of ``act`` without fetching the root tables (use ``choose`` / ``results``).
        ``waves``: run only that many waves (1 on a fresh tree = evaluate and expand the root only,
        TreeSearchT::runPolicyOnly, tree_search.h:387-408); default: the whole move"""
        self.begin_move(active)
        self._pad = int(getattr(actor, "batchsize", 0) or 0)
        for _ in range(self.waves_per_move if waves is None else int(waves)):
            self.wave(actor)
