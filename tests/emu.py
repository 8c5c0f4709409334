"""Test helpers that run the product's C ABI on the SIMT emulator build of the kernel sources
(tests/simt_emu): TEST INFRASTRUCTURE ONLY.  "Device" pointers are host pointers here, so numpy /
CPU torch buffers stand where the CUDA tensors of elf_b200.mcts.MctsBatch are."""
import ctypes
import os
import sys

import numpy as np

from elf_b200 import lib as _l
from elf_b200.board import GoBatch
from elf_b200.refstream import RefStreamSearch

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def emu_lib():
    global _lib
    if _lib is None:
        sys.path.insert(0, os.path.join(_HERE, "simt_emu"))
        import build  # noqa: E402  (tests/simt_emu/build.py)

        _lib = _l.load_library(build.build())  # explicit path: the product loader never picks this up
    return _lib


def emu_batch(G, n):
    """the real GoBatch host class bound to the emulator build"""
    L = emu_lib()
    gb = GoBatch.__new__(GoBatch)
    gb._lib = L
    gb._ctx = _l.vp()
    _l.check(L, L.elfb200_create(n, G, 0, ctypes.byref(gb._ctx)))
    gb.num_games, gb.board_size, gb.num_actions, gb.device, gb._children = G, n, n * n + 1, 0, []
    return gb


class EmuSearch(RefStreamSearch):
    """MctsBatch's interface (begin_move / select / leaf_info / expand_backup / results / choose /
    advance / reset / search / act) over the emulated C ABI with CPU torch tensors"""

    def __init__(self, gb, feature_format="f32", cpad=24, strict_root=True, **opts):
        import torch

        self.feature_format, self.cpad, self.strict_root, self._mismatches = feature_format, int(cpad), strict_root, 0
        self._torch = torch
        self.gb = gb
        self._lib = L = emu_lib()
        o = _l.MctsOptions()
        _l.check(L, L.elfb200_mcts_default_options(ctypes.byref(o)))
        for k, v in opts.items():
            if not hasattr(o, k):
                raise TypeError(f"unknown MCTS option {k}")
            setattr(o, k, v)
        self.options = o
        self._m = _l.vp()
        _l.check(L, L.elfb200_mcts_create(gb._ctx, ctypes.byref(o), ctypes.byref(self._m)))
        n = gb.board_size
        self.waves_per_move = L.elfb200_mcts_waves_per_move(self._m)
        self.max_leaves = L.elfb200_mcts_max_leaves(self._m)
        if feature_format == "f32":
            self._fmt = _l.FEAT_F32_NCHW
            self.feat = torch.zeros((self.max_leaves, 18, n, n), dtype=torch.float32)
        else:
            self._fmt = _l.FEAT_F16_NHWC if feature_format == "f16" else _l.FEAT_BF16_NHWC
            self.feat = torch.zeros((self.max_leaves, n, n, self.cpad),
                                    dtype=torch.float16 if feature_format == "f16" else torch.bfloat16)
        self.feat_key = "s" if feature_format == "f32" else "s_nhwc"
        self.device = torch.device("cpu")
        self._n = 0

    def close(self):
        if self._m:
            self._lib.elfb200_mcts_destroy(self._m)
            self._m = None

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
                self._mismatches = bad
                raise _l.ElfB200Error("TreeSearch::Root state is not the same as the input state")

    def select(self, wait=True):
        k = ctypes.c_int32()
        _l.check(self._lib, self._lib.elfb200_mcts_select_ex(self._m, self.feat.data_ptr(), self._fmt, self.cpad,
                                                             ctypes.byref(k) if wait else None))
        self._n = k.value if wait else -1
        return self.feat[: k.value] if wait else self.feat

    def leaf_count(self):
        k = ctypes.c_int32()
        _l.check(self._lib, self._lib.elfb200_mcts_leaf_count(self._m, ctypes.byref(k)))
        self._n = k.value
        return k.value

    def leaf_info(self):
        n = self._n if self._n >= 0 else self.leaf_count()
        h, g, p = np.empty(n, np.uint64), np.empty(n, np.int32), np.empty(n, np.int32)
        self.leaf_d4 = np.empty(n, np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_leaf_info(self._m, h.ctypes.data, g.ctypes.data, p.ctypes.data,
                                                             self.leaf_d4.ctypes.data))
        return h, g, p

    def expand_backup(self, pi, v):
        if self._n != 0:
            pi = pi.to(self._torch.float32).contiguous()
            v = v.to(self._torch.float32).reshape(-1).contiguous()
            assert pi.shape[0] >= (self._n if self._n > 0 else self.max_leaves)
            _l.check(self._lib, self._lib.elfb200_mcts_expand_backup(self._m, pi.data_ptr(), v.data_ptr()))
        else:
            _l.check(self._lib, self._lib.elfb200_mcts_expand_backup(self._m, None, None))

    def results(self):
        G, P1 = self.gb.num_games, self.gb.num_actions
        best, vis = np.empty(G, np.int32), np.empty((G, P1), np.int32)
        rv, bq, tot = np.empty(G, np.float32), np.empty(G, np.float32), np.empty(G, np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_results(self._m, best.ctypes.data, vis.ctypes.data, rv.ctypes.data,
                                                           bq.ctypes.data, tot.ctypes.data))
        return {"best_action": best, "visits": vis, "root_value": rv, "best_q": bq, "total_visits": tot}

    def choose(self, policy_distri_cutoff, resign_thres, never_resign=None, seed=0):
        G = self.gb.num_games
        a, v = np.empty(G, np.int32), np.empty(G, np.float32)
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
        o = np.empty((self.gb.num_games, self.gb.num_actions), np.float32)
        _l.check(self._lib, self._lib.elfb200_mcts_root_priors(self._m, o.ctypes.data))
        return o

    def errors(self):
        e = np.zeros(4, np.int32)
        _l.check(self._lib, self._lib.elfb200_mcts_errors(self._m, e.ctypes.data))
        return e

    def eval_count(self):
        return self._lib.elfb200_mcts_eval_count(self._m)

    def stats(self):
        s = np.zeros(4, np.uint64)
        _l.check(self._lib, self._lib.elfb200_mcts_stats(self._m, s.ctypes.data))
        return s

    def timings(self, reset=False):
        ms = np.zeros(4, np.float64)
        w = ctypes.c_int64()
        _l.check(self._lib, self._lib.elfb200_mcts_timings(self._m, ms.ctypes.data, ctypes.byref(w), int(reset)))
        return ms, w.value

    def search(self, actor, active=None, waves=None):
        self.begin_move(active)
        for _ in range(self.waves_per_move if waves is None else int(waves)):
            s = self.select()
            if s.shape[0] > 0:
                r = actor({self.feat_key: s})
                self.expand_backup(r["pi"], r["V"])
            else:
                self.expand_backup(None, None)

    def act(self, actor, active=None):
        self.search(actor, active)
        return self.results()
