#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the self-play hot path.

Default workload (BASELINE.json configs[2]; with N GPUs configs[3]): 4096 concurrent 19x19 self-play
games in total (4096/N per GPU), 800 MCTS rollouts per move in waves of 8 per game, random-init
20-block x 256-channel policy/value net in fp16 at NN batch 256, puct 1.5, virtual loss 1, persistent
tree.  One "step" = one search wave of every game in steady state (8 rollouts per game: descents,
leaf features, network, expansion, backup); a move is 100 waves, so
    moves/sec = steps/sec x games x 8 / 800.
Move boundaries that fall inside the timed region (choice, GoState::forward, tree advance) are
timed with it.

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU search driving the
                                                           # same GPU network, all host threads
  python bench.py --workload playout ...                   # configs[1]/[4]: random-policy playouts only

`value`    device-timed (CUDA events spanning all streams), fast path: leaf features stay on the GPU
           as fp16 NHWC, two half batches interleaved so the network stream never drains.
`e2e`      the same metric through the reference's tensor boundary with HOST buffers: float32 "s"
           lands in pinned host memory, the callback moves it to the GPU, pi/V return through pinned
           host memory (src_py/elf/utils_elf.py:39-47,378-405), wall clock.
`roofline` our HBM-bound kernel of this workload, k_leaf_features (SURVEY 8d: 26,792 B/position),
           timed alone; `rooflines` lists the other kernels, the select kernel with its measured DRAM
           bytes next to the 8d formula.  `board_step` is the playout workload with its own roofline.
`cpu_baseline` the compiled reference search (oracle/_ref) on the host cores driving the same network.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

BOARD = 19
GAMES_PER_GPU = 4096
SEED = 20260922
ALGO_BYTES_PER_PLY = 264 + 184  # SURVEY.md 8d: step + legal mask, 19x19 (9x9: 2*(32+32)+8 + 32+32+24 = 224)


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture, or None"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))[kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, rank=0, world=1):
    """--dump-outputs: write what the timed path returned in its last step as ``<out_dir>/<name>.npy``.
    Every array has one row per game; integers are stored as float64 (exact up to 2**53), 64-bit hashes
    as two 32-bit halves.  When the rows exceed DUMP_LIMIT_BYTES a fixed, seeded sample of games is kept
    (``game_index.npy`` names the rows in every case), so two builds can be compared file by file."""
    conv = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype == np.uint64:
            conv[name + "_hi"] = (a >> np.uint64(32)).astype(np.float64)
            conv[name + "_lo"] = (a & np.uint64(0xFFFFFFFF)).astype(np.float64)
        elif a.dtype.kind in "iub":
            conv[name] = a.astype(np.float64)
        else:
            conv[name] = a.astype(np.float32)
    G = len(next(iter(conv.values())))
    row_bytes = sum(a[:1].nbytes for a in conv.values()) + 8
    keep = np.arange(G)
    if G * row_bytes > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(SEED).choice(G, DUMP_LIMIT_BYTES // row_bytes, replace=False))
    conv["game_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in conv.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a if name == "game_index" else a[keep])


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (oracle/_ref) or the oracle port, all host threads
# --------------------------------------------------------------------------------------------
def effective_cores():
    """host threads this process can really use: affinity mask capped by the cgroup CPU quota"""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def cpu_playouts(seconds=None, games_per_thread=None, first_id=10_000_000):
    """Run random-policy playouts on every host core.  Either time-bounded (`seconds`) or a fixed
    number of games per thread.  Returns dict(moves, seconds, cores, kind, games)."""
    from tests import oracles

    cores = effective_cores()
    if oracles.have_ref(BOARD):
        kind = "reference"
        L = oracles.load_ref(BOARD)

        def one(gid):
            chk = ctypes.c_uint64()
            sc = ctypes.c_int32()
            return L.ref_playout(SEED, gid, 2 * BOARD * BOARD, None, None, None, ctypes.byref(chk), ctypes.byref(sc))
    else:
        kind = "port"
        L = oracles.load_oracle()

        def one(gid):
            chk = ctypes.c_uint64()
            sc = ctypes.c_int32()
            return L.go_playout(BOARD, SEED, gid, 2 * BOARD * BOARD, None, None, None, ctypes.byref(chk), ctypes.byref(sc))

    moves = [0] * cores
    games = [0] * cores
    t0 = time.perf_counter()
    deadline = t0 + seconds if seconds else None

    def work(tid):
        gid = first_id + tid * 1_000_000
        n = 0
        while True:
            if deadline is not None and time.perf_counter() >= deadline:
                break
            if games_per_thread is not None and n >= games_per_thread:
                break
            moves[tid] += one(gid + n)  # ctypes releases the GIL during the call
            n += 1
        games[tid] = n

    th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
    [t.start() for t in th]
    [t.join() for t in th]
    dt = time.perf_counter() - t0
    return {"moves": sum(moves), "seconds": dt, "cores": cores, "kind": kind, "games": sum(games)}


def run_reference_playout(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    gpt = 24  # games per thread per step: ~0.15-0.3 s of CPU work per step
    for _ in range(args.warmup):
        cpu_playouts(games_per_thread=4)
    tot_moves, tot_s, info = 0, 0.0, None
    for _ in range(args.steps):
        info = cpu_playouts(games_per_thread=gpt)
        tot_moves += info["moves"]
        tot_s += info["seconds"]
    val = tot_moves / tot_s
    sample = f"{gpt} playouts/thread/step x {info['cores']} threads (of the 4096-game batch), {args.steps} steps"
    line = {
        "impl": "reference", "metric": f"self-play moves/sec (random-policy playouts, {BOARD}x{BOARD})", "value": val,
        "unit": "moves/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": f"configs[1]: {args.games} concurrent {BOARD}x{BOARD} games, random-policy playouts (each host thread plays games back to back)",
                   "games_per_gpu": args.games, "board": BOARD, "seed": SEED},
        "cpu_baseline": {"value": val, "unit": "moves/s", "cores": info["cores"], "kind": info["kind"], "sample": sample},
        "e2e": {"value": val, "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# --------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def run_playout(args):
    import torch

    import elf_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    G = args.games
    gb = elf_b200.GoBatch(G, board_size=BOARD, device=local)
    eff_layout = args.playout_layout if args.playout_layout >= 0 else (1 if (BOARD == 19 and G >= 12288) else 0)
    gb.set_playout_layout(eff_layout)
    stream = torch.cuda.ExternalStream(gb.stream, device=local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")  # > 126 MB L2

    from elf_b200.dist_utils import reduce_timing_and_counts, shard_first_game_id

    def first_id(step):  # distinct games per (step, rank)
        return shard_first_game_id(step, world, rank, G)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    PLIES = args.plies_per_slot

    # ---- warm-up -----------------------------------------------------------------------------
    for w in range(args.warmup):
        gb.playout_stream_launch(SEED, first_id(10_000 + w), PLIES)
    gb.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    # ---- device-timed region: K steps, CUDA events on the library's stream, L2 flushed between --
    launches0 = gb.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    plies_total = 0
    barrier()
    t_wall0 = time.perf_counter()
    for s in range(args.steps):
        with torch.cuda.stream(stream):
            flush.fill_(s & 0xFF)  # evict L2 (outside the event pair)
            ev[s][0].record(stream)
        gb.playout_stream_launch(SEED, first_id(s), PLIES)
        with torch.cuda.stream(stream):
            ev[s][1].record(stream)
        gb.synchronize()
        plies_total += gb.playout_results()["total_plies"]
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = gb.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    if args.dump_outputs:
        r = gb.playout_results()  # what playout_stream() returns: in this mode "score" holds the games started
        dump_outputs(args.dump_outputs, {"chk": r["chk"], "plies": r["plies"], "games": r["score"], "hash": r["hash"]},
                     rank, world)

    # ---- e2e: the public call with host result buffers, wall clock ------------------------------
    barrier()
    t0 = time.perf_counter()
    e2e_plies = 0
    for s in range(args.steps):
        r = gb.playout_stream(SEED, first_id(s), PLIES)  # launch + D2H(chk, plies, games, hash) + sync
        e2e_plies += r["total_plies"]
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- secondary: one batch of G games played to terminal (includes the ragged tail) -----------
    tt_ms, tt_plies = 0.0, 0
    for s in range(min(args.steps, 10)):
        a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            a.record(stream)
        gb.playout_launch(SEED, first_id(s))
        with torch.cuda.stream(stream):
            b2.record(stream)
        gb.synchronize()
        tt_ms += a.elapsed_time(b2)
        tt_plies += gb.playout_results()["total_plies"]
    clocks = sampler.stop() if rank == 0 else None

    # ---- secondary: the step API (GoState::forward for the whole batch per call, HOST buffers) --------
    step_api = None
    if rank == 0:
        try:
            gold = json.load(open(os.path.join(ROOT, "tests", "golden", f"playouts_{BOARD}.json")))
            mv = next(e["moves"] for e in gold["games"] if "moves" in e)
            gb.reset()
            acts = np.empty(G, np.int32)
            gb.forward(np.full(G, mv[0], np.int32))
            gb.reset()
            t_s = time.perf_counter()
            for a in mv:
                acts.fill(a)
                ok = gb.forward(acts)  # H2D actions, k_step, D2H accept flags, sync
            dt_s = time.perf_counter() - t_s
            step_api = {"value": G * len(mv) / dt_s, "unit": "moves/s", "us_per_call": 1e6 * dt_s / len(mv),
                        "all_accepted": bool(ok.all()), "h2d_bytes_per_call": 4 * G, "d2h_bytes_per_call": G,
                        "note": "elfb200_step(): every game replays one reference move list, one call per ply"}
        except Exception as e:
            step_api = f"unmeasured: {e}"

    # ---- spot parity of timed work (rank 0): a few games of step 0 against the oracle ------------
    parity = None
    if rank == 0:
        try:
            from tests import oracles

            r0 = gb.playout_stream(SEED, first_id(0), PLIES)
            ok = True
            for g in (0, 1337, G - 1):
                t, acc, games = oracles.oracle_playout_stream(BOARD, SEED, first_id(0), g, G, PLIES)
                ok &= (t, acc, games) == (int(r0["plies"][g]), int(r0["chk"][g]), int(r0["games"][g]))
            parity = bool(ok)
        except Exception as e:  # oracle missing is not fatal for the bench
            parity = f"unchecked: {e}"

    # ---- reduce over ranks (MAX of times, SUM of counters) ----------------------------------------
    (dev_ms, e2e_s), (plies_total, e2e_plies, launches) = reduce_timing_and_counts(
        dist, f"cuda:{local}", [dev_ms, e2e_s], [plies_total, e2e_plies, launches])

    if rank == 0:
        peak, peak_src = measured_peaks()
        value = plies_total / (dev_ms / 1e3)
        per_rank_plies = plies_total / world
        algo = ALGO_BYTES_PER_PLY if BOARD == 19 else 224
        achieved = algo * per_rank_plies / args.steps / (dev_ms / args.steps / 1e3) / 1e9
        line = {
            "metric": f"self-play moves/sec (random-policy playouts, {BOARD}x{BOARD})", "value": value, "unit": "moves/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": (f"configs[1]: 4096 concurrent 19x19 games per GPU" if (BOARD, G) == (19, 4096) else f"configs[4]-style: {G} concurrent {BOARD}x{BOARD} games per GPU") + f", random-policy playouts, steady state: every game slot plays {PLIES} plies per step and restarts finished games",
                       "games_per_gpu": G, "board": BOARD, "seed": SEED, "plies_per_step": plies_total / args.steps,
                       "plies_per_slot": PLIES,
                       "l2": "flushed (256 MiB write) between timed steps", "parallelism": f"games sharded x{world}, no collective"},
            "e2e": {"value": e2e_plies / e2e_s, "unit": "moves/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 24 * G,
                    "note": "elfb200_playout_stream() from the host, results read back every step; this workload's inputs are 3 scalars "
                            "(seed, first id, plies per slot) passed as kernel params, so there is nothing to copy in.  The host-driven "
                            "flavour of the same path -- one elfb200_step() per ply with HOST action and accept buffers -- is in host_driven",
                    "host_driven": step_api if isinstance(step_api, dict) else {"unmeasured": str(step_api)}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": measured_traffic("k_playout<19>") if BOARD == 19 else None, "peak_source": peak_src,
                         "kernel": f"k_playout{2 if eff_layout else ''}<{BOARD}>", "algorithmic_bytes_per_ply": algo,
                         "note": "position and group masks live in registers, the superko record in L2: DRAM is idle and the kernel is bound by the integer ALU pipe (profiles/r1_playout_F.md)"},
            "clocks": clocks, "wall_s_timed_region": t_wall, "parity_spot_check": parity, "step_api": step_api,
            "batch_to_terminal": {"value": tt_plies / (tt_ms / 1e3) * 1.0, "unit": "moves/s (this rank)",
                                  "ms_per_batch": tt_ms / max(1, min(args.steps, 10)),
                                  "note": "one batch of 4096 games from the empty board to terminated(): includes the ragged tail"},
        }
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_playouts(seconds=args.cpu_seconds)
            line["cpu_baseline"] = {
                "value": cb["moves"] / cb["seconds"], "unit": "moves/s", "cores": cb["cores"], "kind": cb["kind"],
                "sample": f"{cb['games']} playouts of the same workload in {cb['seconds']:.1f} s on {cb['cores']} threads"}
        emit(line)
    gb.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# --------------------------------------------------------------------------------------------
# headline workload: BASELINE configs[2]/[3] -- MCTS self-play.  The network is PyTorch/cuDNN plumbing
# (elf_b200.model.FusedActor); our kernels are select / leaf features / expand / backup / choose /
# step / advance.
# --------------------------------------------------------------------------------------------
ROLLOUTS, PER_BATCH, NN_BATCH = 800, 8, 256
ISSUE_SLOTS_PER_S = 148 * 4  # x SM clock: warp instructions the chip can issue per second


def load_profile_numbers():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def make_network(args, dev):
    """the 20x256 policy/value net of configs[2] (random init, fixed seed) behind the model-interface
    callback; returns (actor, description, module)"""
    import torch

    from elf_b200.model import FusedActor, PolicyValueNet

    torch.manual_seed(1234)
    if args.fake_net:
        P1 = BOARD * BOARD + 1
        table = torch.rand(4096, P1, device=dev).softmax(1)
        vals = torch.rand(4096, device=dev) * 2 - 1

        def actor(batch):
            n = (batch["s"] if "s" in batch else batch["s_nhwc"]).shape[0]
            idx = torch.arange(n, device=dev) % 4096
            return {"pi": table[idx], "V": vals[idx]}
        return actor, "fake (table lookup: engine-only timing, BASELINE.md config 3a)", None
    torch.backends.cudnn.benchmark = True
    model = PolicyValueNet(BOARD, num_block=args.blocks, dim=args.dim).to(dev).eval()
    return None, (f"random-init resnet {args.blocks}x{args.dim} (df_model3.Model_PolicyValue), fp16, BatchNorm folded, "
                  f"cuDNN fused conv+bias(+add)+ReLU, NN batch {args.nn_batch} replayed as a CUDA graph"), model


def random_opening(gb, plies, rng):
    """`plies` uniformly random legal non-pass moves in every game (host-chosen from the legal masks)"""
    import numpy as np

    for _ in range(plies):
        lg = gb.legal_mask()[:, :-1].astype(np.float64)
        lg += 1e-9  # a game without a legal point would pass below
        lg /= lg.sum(1, keepdims=True)
        c = lg.cumsum(1)
        a = (c < rng.random((lg.shape[0], 1))).sum(1).astype(np.int32)
        a = np.minimum(a, lg.shape[1] - 1)
        ok = gb.forward(a)
        if not ok.all():  # the epsilon picked an illegal point somewhere: those games pass instead
            a2 = np.where(ok, -1, BOARD * BOARD).astype(np.int32)
            gb.forward(a2)


class HostBoundary:
    """The reference's tensor boundary around the model callback (utils_elf.py:39-47,378-405): the
    feature batch lands in PINNED HOST memory, the callback moves it to the GPU, and the replies go back
    through pinned host memory.  Used for the `e2e` reading; counts the bytes it moves."""

    def __init__(self, actor, rows, n, dev):
        import torch

        self.actor, self.dev = actor, dev
        self.batchsize = getattr(actor, "batchsize", 0)
        self.s = torch.empty((rows, 18, n, n), dtype=torch.float32, pin_memory=True)
        self.pi = torch.empty((rows, n * n + 1), dtype=torch.float32, pin_memory=True)
        self.v = torch.empty((rows,), dtype=torch.float32, pin_memory=True)
        self.h2d = self.d2h = 0

    def __call__(self, batch):
        import torch

        s = batch["s"]
        m = s.shape[0]
        self.s[:m].copy_(s, non_blocking=True)  # D2H: what GoFeature's extractor + SharedMem do in the reference
        torch.cuda.current_stream(self.dev).synchronize()
        x = self.s[:m].to(self.dev, non_blocking=True)  # H2D: the callback's .cuda()
        out = self.actor({"s": x})
        self.pi[:m].copy_(out["pi"], non_blocking=True)  # D2H: reply tensors are host tensors
        self.v[:m].copy_(out["V"].reshape(-1), non_blocking=True)
        torch.cuda.current_stream(self.dev).synchronize()
        self.d2h += m * (18 * s.shape[2] * s.shape[3] + self.pi.shape[1] + 1) * 4
        self.h2d += m * (18 * s.shape[2] * s.shape[3] + self.pi.shape[1] + 1) * 4
        return {"pi": self.pi[:m].to(self.dev, non_blocking=True), "V": self.v[:m].to(self.dev, non_blocking=True)}


class SelfPlayEngine:
    """G games on one GPU as `parts` SelfPlay batches driven wave by wave through a WavePipeline"""

    def __init__(self, actor, G, parts, local, rank, feature_format, opening_plies=16):
        import numpy as np

        import elf_b200
        from elf_b200.pipeline import WavePipeline

        sizes = [G // parts + (1 if i < G % parts else 0) for i in range(parts)]
        self.sp = [elf_b200.selfplay.SelfPlay(
            actor, num_games=g, board_size=BOARD, device=local, policy_distri_cutoff=0, resign_thres=0.0,
            never_resign_ratio=1.0, num_rollouts=ROLLOUTS, num_rollouts_per_batch=PER_BATCH, virtual_loss=1,
            persistent_tree=1, c_puct=1.5, rotation_flip=1, seed=rank * 16 + i, feature_format=feature_format)
            for i, g in enumerate(sizes) if g > 0]
        rng = np.random.default_rng(99 + rank)
        for sp in self.sp:
            random_opening(sp.gb, opening_plies, rng)
        self.actor = actor
        self.pipe = WavePipeline([sp.mcts for sp in self.sp], actor)
        self.wpm = self.pipe.waves_per_move
        self.wave_in_move = 0
        self.moves = 0
        self.infos = None

    def _begin(self):
        self.infos = [sp.gb.info() for sp in self.sp]
        self.pipe.begin_move()
        self.wave_in_move = 0

    def step(self, pipelined=True, actor=None):
        """one wave of every game; at a move boundary also the move itself"""
        if self.infos is None:
            self._begin()
        if pipelined:
            self.pipe.waves(1)
        else:
            self.pipe.drain()
            for sp in self.sp:
                sp.mcts._pad = int(getattr(actor or self.actor, "batchsize", 0) or 0)
                sp.mcts.wave(actor or self.actor)
        self.wave_in_move += 1
        if self.wave_in_move == self.wpm:
            self.pipe.drain()
            for sp, info in zip(self.sp, self.infos):
                self.moves += sp.finish_move(info)
            self._begin()

    def set_feature_format(self, fmt):
        self.pipe.drain()
        for sp in self.sp:
            sp.mcts.set_feature_format(fmt)

    def launches(self):
        return sum(sp.gb.launch_count() for sp in self.sp)

    def evals(self):
        return sum(sp.mcts.eval_count() for sp in self.sp)

    def errors(self):
        import numpy as np

        return np.sum([sp.mcts.errors() for sp in self.sp], axis=0)

    def streams(self):
        import torch

        return [torch.cuda.ExternalStream(sp.gb.stream, device=self.pipe.device) for sp in self.sp] + [self.pipe.nn_stream]

    def close(self):
        self.pipe.drain()
        for sp in self.sp:
            sp.close()


def device_span(streams, fn):
    """run fn() and return the device time (ms) from 'all streams idle' to 'all streams done'"""
    import torch

    torch.cuda.synchronize()
    cur = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    for st in streams:
        st.wait_event(e0)
    fn()
    for st in streams:
        cur.wait_stream(st)
    e1.record(cur)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def board_step_probe(local, steps=10, warmup=3, G=4096, plies=512, layout=0):
    """BASELINE's second metric, "board-step GB/s vs roofline": the configs[1] playout workload (4096
    concurrent games, steady state) timed on its own, with the HBM formula AND the issue-slot roof"""
    import torch

    import elf_b200

    gb = elf_b200.GoBatch(G, board_size=BOARD, device=local)
    gb.set_playout_layout(layout)
    stream = torch.cuda.ExternalStream(gb.stream, device=local)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local}")
    for w in range(warmup):
        gb.playout_stream_launch(SEED, 10_000_000 + w * G, plies)
    gb.synchronize()
    ms, tot = 0.0, 0
    for s in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            flush.fill_(s & 0xFF)
            a.record(stream)
        gb.playout_stream_launch(SEED, s * G, plies)
        with torch.cuda.stream(stream):
            b.record(stream)
        gb.synchronize()
        ms += a.elapsed_time(b)
        tot += gb.playout_results()["total_plies"]
    # the host-driven flavour of the board step: one elfb200_step() per ply with HOST action / accept buffers
    # (GoState::forward for the whole batch per call; zero-copy mapped window, one launch + one wait)
    host = None
    try:
        import numpy as np

        gold = json.load(open(os.path.join(ROOT, "tests", "golden", f"playouts_{BOARD}.json")))
        mv = next(e["moves"] for e in gold["games"] if "moves" in e)
        acts = np.empty(G, np.int32)
        gb.reset()
        gb.forward(np.full(G, mv[0], np.int32))
        gb.reset()
        t0 = time.perf_counter()
        for a_ in mv:
            acts.fill(a_)
            ok = gb.forward(acts)
        dt = time.perf_counter() - t0
        host = {"value": G * len(mv) / dt, "unit": "moves/s", "us_per_call": 1e6 * dt / len(mv), "all_accepted": bool(ok.all()),
                "bytes_per_call_over_pcie": 5 * G,
                "note": "elfb200_step(): every game replays one reference move list, one call per ply, host buffers"}
    except Exception as e:
        host = {"unmeasured": str(e)}
    gb.close()
    peak, peak_src = measured_peaks()
    kname = f"k_playout{2 if layout else ''}<{BOARD}>"
    prof = load_profile_numbers().get(kname, {})
    rate = tot / (ms / 1e3)
    algo = ALGO_BYTES_PER_PLY if BOARD == 19 else 224
    out = {"value": rate, "unit": "moves/s", "workload": f"configs[1]: {G} concurrent {BOARD}x{BOARD} games, random-policy playouts, "
           f"steady state ({plies} plies per slot per step, finished games restart)", "ms_per_step": ms / steps, "steps": steps,
           "roofline": {"bound": "hbm", "achieved": algo * rate / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": algo * rate / 1e9 / peak, "traffic": prof.get("dram_bytes_per_launch"),
                        "peak_source": peak_src, "kernel": kname, "algorithmic_bytes_per_ply": algo,
                        "note": "SURVEY 8d byte formula; the position lives in registers, DRAM is idle -- the honest roof is issue_roof"},
           "lane_layout": "two board rows per lane, three games per warp" if layout else "one board row per lane, one game per warp",
           "host_driven": host}
    wi = prof.get("warp_inst_per_ply")
    if wi:
        try:
            ghz = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"] / 1e3
        except Exception:
            ghz = 1.965
        roof = ISSUE_SLOTS_PER_S * ghz * 1e9 / wi
        out["issue_roof"] = {"warp_inst_per_ply": wi, "plies_per_s_at_full_issue": roof, "frac": rate / roof,
                             "note": "148 SMs x 4 schedulers x SM clock / (warp instructions per game-ply from the committed ncu capture)"}
    return out


def selfplay_config(args, world, net_desc):
    """the `config` object of the bench line: identical for both arms at the same N"""
    G_total = args.games
    moves_per_step = G_total * PER_BATCH / ROLLOUTS
    return {
        "workload": (f"configs[{(2 if world == 1 else 3) if BOARD == 19 else 4}]: {G_total} concurrent {BOARD}x{BOARD} self-play games in total "
                     f"({G_total // world} per GPU), {ROLLOUTS} MCTS rollouts/move in waves of {PER_BATCH}, puct 1.5, "
                     f"virtual loss 1, persistent tree, NN batch {args.nn_batch}; step = one wave of every game "
                     f"(= {moves_per_step:.2f} moves), steady state after {args.opening_plies} random opening plies"),
        "net": net_desc, "games_total": G_total, "games_per_gpu": G_total // world, "rollouts_per_move": ROLLOUTS,
        "rollouts_per_wave": PER_BATCH, "nn_batch": args.nn_batch, "board": BOARD, "parts_per_gpu": args.parts,
        "l2": "inputs larger than L2: the node pool is %.1f GB per GPU and a wave's leaf batch %.0f MB" % (
            (G_total // world) * (2 * ROLLOUTS + 256) * (BOARD * BOARD + 1) * 20.5 / 1e9,
            (G_total // world) * PER_BATCH * BOARD * BOARD * 48 / 1e6),
        "parallelism": f"games sharded x{world}, NCCL weight broadcast only"}


def feature_writer_probe(local, G=32768, reps=10):
    """the board batch's k_features (same CTA code as k_leaf_features, history from the ring) at 32768
    positions: float32 NCHW and fp16 NHWC, CUDA events around back-to-back launches"""
    import numpy as np
    import torch

    import elf_b200
    from elf_b200 import lib as L

    gb = elf_b200.GoBatch(G, board_size=BOARD, device=local)
    dev = torch.device("cuda", local)
    st = torch.cuda.ExternalStream(gb.stream, device=dev)
    rng = np.random.default_rng(5)
    random_opening(gb, 12, rng)
    d4 = torch.from_numpy(rng.integers(0, 8, G).astype(np.int32)).to(dev)
    P = BOARD * BOARD
    o32 = torch.empty((G, 18, BOARD, BOARD), dtype=torch.float32, device=dev)
    o16 = torch.empty((G, BOARD, BOARD, 24), dtype=torch.float16, device=dev)
    peak, _ = measured_peaks()
    out = {}
    for name, fn, byts in (("float32_nchw", lambda: gb.features_dev(o32.data_ptr(), d4.data_ptr()), 800 + 18 * P * 4),
                           ("fp16_nhwc", lambda: gb.features_dev(o16.data_ptr(), d4.data_ptr(), L.FEAT_F16_NHWC, 24), 800 + P * 48)):
        fn()
        gb.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(reps):
            fn()
        b.record(st)
        gb.synchronize()
        ms = a.elapsed_time(b) / reps
        out[name] = {"ms_per_launch": ms, "achieved": G * byts / ms / 1e6, "unit": "GB/s", "peak": peak,
                     "frac": G * byts / ms / 1e6 / peak, "algorithmic_bytes_per_position": byts}
    gb.close()
    out["note"] = f"k_features<{BOARD}>, {G} positions per launch, {reps} launches back to back (outputs 852 MB / 568 MB: larger than L2)"
    return out


def run_selfplay(args):
    import numpy as np
    import torch

    from elf_b200.model import FusedActor, broadcast_weights

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    G_total = args.games
    G = G_total // world + (1 if rank < G_total % world else 0)  # games sharded, total fixed (configs[3]: 512/GPU at 8)
    actor, net_desc, model = make_network(args, dev)
    t_bcast = 0.0
    if model is not None:
        barrier()
        t0 = time.perf_counter()
        broadcast_weights(model)  # frozen weights from rank 0: the only collective of the path
        torch.cuda.synchronize()
        t_bcast = time.perf_counter() - t0
        actor = FusedActor(model, batchsize=args.nn_batch, dtype=torch.float16, cuda_graph=True)
    def note(msg):
        if rank == 0:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)

    note(f"network ready ({net_desc}); building {G} games in {args.parts} part(s)")
    eng = SelfPlayEngine(actor, G, args.parts, local, rank, "f32" if args.fake_net else "f16", args.opening_plies)
    streams = eng.streams()
    K, W = args.steps, args.warmup
    note("engine ready, warm-up")

    for _ in range(W):
        eng.step()
    eng.pipe.drain()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0, ev0, mv0 = eng.launches(), eng.evals(), eng.moves
    barrier()
    t0 = time.perf_counter()
    dev_ms = device_span(streams, lambda: ([eng.step() for _ in range(K)], eng.pipe.drain()))
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    launches, evals, real_moves = eng.launches() - l0, eng.evals() - ev0, eng.moves - mv0
    note(f"timed region: {K} steps in {dev_ms:.1f} ms device / {wall * 1e3:.1f} ms wall, {evals} evaluations")
    if args.dump_outputs:
        # the root tables MctsBatch.results() hands a caller after the last timed wave, games in batch order
        res = [sp.mcts.results() for sp in eng.sp]
        out = {k: np.concatenate([r[k] for r in res]) for k in ("visits", "root_value", "best_q", "best_action", "total_visits")}
        out["root_priors"] = np.concatenate([sp.mcts.root_priors() for sp in eng.sp])
        dump_outputs(args.dump_outputs, out, rank, world)
        note(f"outputs of the last timed step written to {args.dump_outputs}")

    # ---- e2e: the same waves through the host-buffer tensor boundary (float32 "s"), wall clock --------
    Ke = min(K, args.e2e_steps)
    e2e_s, hb_h2d, hb_d2h, e2e_err = None, 0, 0, None
    try:
        eng.set_feature_format("f32")
        hb = HostBoundary(actor, max(sp.mcts.max_leaves for sp in eng.sp), BOARD, dev)
        eng.step(pipelined=False, actor=hb)  # warm (pinned buffers, eager shapes)
        hb.h2d = hb.d2h = 0
        barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            eng.step(pipelined=False, actor=hb)
        barrier()
        e2e_s = time.perf_counter() - t0
        hb_h2d, hb_d2h = hb.h2d / Ke, hb.d2h / Ke
        note(f"e2e (host-buffer boundary): {Ke} steps in {e2e_s * 1e3:.1f} ms wall")
        del hb
    except Exception as e:  # never lose the device-timed line over the secondary reading
        e2e_err = repr(e)
        note("e2e phase failed: " + e2e_err)
        if dist is not None:
            raise

    # ---- kernel timings, alone (no overlap with the network): CUDA events inside the library ---------
    # The feature writer is timed as 10 back-to-back launches on the same pending leaves (idempotent), so
    # the event pair brackets a busy stream and excludes launch latency.
    def time_kernels():
        kern = {}
        for fmt in ("f32", "f16"):
            if args.fake_net and fmt != "f32":
                continue
            eng.set_feature_format(fmt)
            for sp in eng.sp:
                sp.mcts.timings(reset=True)
            st0 = np.sum([sp.mcts.stats().astype(np.int64) for sp in eng.sp], axis=0)
            e0 = eng.evals()
            feat_ms, feat_pos, feat_launches = 0.0, 0, 0
            for _ in range(3):
                if eng.infos is None:
                    eng._begin()
                eng.pipe.drain()
                for sp in eng.sp:
                    mc = sp.mcts
                    mc._pad = int(getattr(eng.actor, "batchsize", 0) or 0)
                    torch.cuda.synchronize()  # nothing else on the GPU: the other part's network batch has drained
                    s_ = mc.wave_select()
                    if s_ is not None:
                        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a_.record(mc._stream)
                        for _r in range(10):
                            mc.leaf_features_again()
                        b_.record(mc._stream)
                        sp.gb.synchronize()
                        feat_ms += a_.elapsed_time(b_)
                        feat_pos += 10 * mc._n
                        feat_launches += 10
                    mc.wave_finish(mc.wave_eval(eng.actor, s_))
                    torch.cuda.synchronize()
                eng.wave_in_move += 1
                if eng.wave_in_move == eng.wpm:
                    eng.pipe.drain()
                    for sp, info in zip(eng.sp, eng.infos):
                        eng.moves += sp.finish_move(info)
                    eng._begin()
            eng.pipe.drain()
            ms = np.sum([sp.mcts.timings()[0] for sp in eng.sp], axis=0)
            waves = eng.sp[0].mcts.timings()[1]
            st = np.sum([sp.mcts.stats().astype(np.int64) for sp in eng.sp], axis=0) - st0
            kern[fmt] = {"ms": ms, "waves": waves, "stats": st, "evals": eng.evals() - e0,
                         "feat_ms": feat_ms, "feat_pos": feat_pos, "feat_launches": feat_launches}
        return kern

    kern = None
    if rank == 0:
        try:
            kern = time_kernels()
        except Exception as e:
            note("kernel timing phase failed: " + repr(e))
    errs = eng.errors()
    eng.close()
    del eng
    torch.cuda.empty_cache()

    note("kernel timings done; board-step probe")
    board = None
    if rank == 0 and not args.no_board_step:
        try:  # a secondary reading must never cost the headline line
            board = board_step_probe(local, layout=max(args.playout_layout, 0))
            if BOARD == 19:
                # the same kernel family where it is issue-bound rather than latency-bound: 16384 games, two rows per lane
                big = board_step_probe(local, steps=4, warmup=3, G=16384, layout=1)
                board["at_16384_games_two_rows_per_lane"] = {k: big[k] for k in ("value", "unit", "ms_per_step", "lane_layout")}
        except Exception as e:
            board = {"unmeasured": repr(e)} if board is None else dict(board, at_16384_games_two_rows_per_lane={"unmeasured": repr(e)})
    featw = None
    if rank == 0 and not args.no_board_step:
        try:
            featw = feature_writer_probe(local)
        except Exception as e:
            featw = {"unmeasured": repr(e)}

    # ---- reduce over ranks (MAX of times, SUM of counters) ----------------------------------------------
    if dist is not None:
        t = torch.tensor([dev_ms, wall, e2e_s or 0.0, t_bcast], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall, e2e_s, t_bcast = t.tolist()
        c = torch.tensor([launches, evals, real_moves, int(errs[1]), int(errs[3])], dtype=torch.int64, device=dev)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        launches, evals, real_moves, e1, e3 = c.tolist()
        errs = [int(errs[0]), e1, int(errs[2]), e3]
    if rank == 0:
        peak, peak_src = measured_peaks()
        prof = load_profile_numbers()
        moves_per_step = G_total * PER_BATCH / ROLLOUTS
        value = K * moves_per_step / (dev_ms / 1e3)
        line = {
            "metric": "self-play moves/sec (MCTS, 19x19)", "value": value, "unit": "moves/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32 search statistics / fp16 network", "data": "synthetic",
            "config": selfplay_config(args, world, net_desc),
            "e2e": {"value": (Ke * moves_per_step / e2e_s) if e2e_s else None, "unit": "moves/s", "steps": Ke, "error": e2e_err,
                    "h2d_bytes_per_step": int(hb_h2d), "d2h_bytes_per_step": int(hb_d2h),
                    "note": "same waves through the reference's tensor boundary with HOST buffers: float32 s -> pinned host -> GPU -> "
                            "network -> pi/V -> pinned host -> GPU (rank 0's bytes per step), wall clock, no overlap between parts"},
            "gpu_launches": int(launches), "nn_evals": int(evals), "nn_positions_per_s": evals / (dev_ms / 1e3),
            "moves_completed_in_timed_region": int(real_moves),
            "weight_broadcast_s": t_bcast, "wall_s_timed_region": wall,
            "host_gap_ms_per_step": max(0.0, (wall * 1e3 - dev_ms) / K),
            "search_errors": {"root_mismatch": int(errs[0]), "pool_overflow": int(errs[1]), "depth_cut": int(errs[2]),
                              "tree_prunes": int(errs[3])},
            "clocks": clocks,
        }
        if kern:
            line.update(kernel_rooflines(kern, prof, peak, peak_src, args.parts))
        else:
            line["roofline"] = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
                                "kernel": f"k_leaf_features<{BOARD}>", "note": "kernel timing phase did not run (see stderr)"}
        if board is not None:
            line["board_step"] = board
        if featw is not None:
            line.setdefault("rooflines", {})["k_features_board_batch"] = featw
        if world == 1 and not args.no_cpu_baseline and not args.fake_net:
            note("cpu_baseline: reference search on the host cores")
            try:
                line["cpu_baseline"] = ref_selfplay(actor, dev, steps=args.cpu_steps, warmup=1)
            except Exception as e:
                line["cpu_baseline"] = {"unavailable": repr(e)}
        if world == 1 and not args.no_cpu_baseline and args.fake_net:
            try:
                line["cpu_baseline"] = ref_selfplay_fake_net(min(args.cpu_seconds, 15.0))
            except Exception as e:
                line["cpu_baseline"] = {"unavailable": repr(e)}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def kernel_rooflines(kern, prof, peak, peak_src, parts):
    """roofline objects from the kernels timed alone (3 waves, CUDA events in the library)"""
    out = {"rooflines": {}}
    k32 = kern["f32"]
    w = max(int(k32["waves"]), 1)
    ms, st, ev = k32["ms"], k32["stats"], k32["evals"]
    P = BOARD * BOARD
    hist_bytes = 8 * 2 * 8 * ((P + 63) // 64) + 32  # SURVEY 8d: 8 history pairs of packed colour bitboards + meta
    feat_bytes = hist_bytes + 18 * P * 4  # + 18 float32 planes: 26,792 B at 19x19
    kq = f"<{BOARD}>"
    feat_gbs = k32["feat_pos"] * feat_bytes / (k32["feat_ms"] / 1e3) / 1e9 if k32["feat_ms"] > 0 else 0.0
    traffic = prof.get("k_leaf_features" + kq, {}).get("dram_bytes_per_launch")
    out["roofline"] = {"bound": "hbm", "achieved": feat_gbs, "peak": peak, "unit": "GB/s", "frac": feat_gbs / peak,
                       "traffic": traffic, "peak_source": peak_src, "kernel": f"k_leaf_features{kq} (float32 NCHW, the GoFeature contract)",
                       "algorithmic_bytes_per_position": feat_bytes,
                       "positions_per_launch": k32["feat_pos"] / max(k32["feat_launches"], 1),
                       "ms_per_launch": k32["feat_ms"] / max(k32["feat_launches"], 1),
                       "note": "CUDA events around 10 back-to-back launches on the pending leaves of a wave (idempotent), GPU "
                               "otherwise idle, 3 waves x parts; a launch covers one part's leaves (their 8-position histories "
                               "were laid out contiguously by k_select when it claimed them)"}
    sel_formula = int(st[0]) * (32 + 4) + int(st[3]) * 16  # SURVEY 8d: header + E_n*16 + vl write (full scan)
    sel_prefix = int(st[0]) * (32 + 4) + int(st[1]) * 16   # what the prefix scan touches
    sel_ms = ms[0]
    sel = {"bound": "hbm", "kernel": "k_select" + kq, "unit": "GB/s", "peak": peak,
           "formula_GBps": sel_formula / (sel_ms / 1e3) / 1e9, "prefix_scan_GBps": sel_prefix / (sel_ms / 1e3) / 1e9,
           "ms_per_wave": sel_ms / w, "nodes_visited": int(st[0]), "edges_scanned": int(st[1]), "edges_stored": int(st[3])}
    dsel = prof.get("k_select" + kq, {}).get("dram_bytes_per_launch")
    if dsel and prof.get("k_select" + kq, {}).get("launch_ms"):
        p = prof["k_select" + kq]
        sel["measured_dram_GBps"] = p["dram_bytes_per_launch"] / (p["launch_ms"] / 1e3) / 1e9
        sel["achieved"] = sel["measured_dram_GBps"]
        sel["frac"] = sel["measured_dram_GBps"] / peak
        sel["note"] = ("frac is MEASURED DRAM bytes / time from the committed ncu capture (profiles/), not the 8d full-scan "
                       "formula: the kernel reads only the selected prefix of each node's edges and is bound by the "
                       "dependent-load latency of the descent, not by bandwidth")
    else:
        sel["achieved"] = sel["prefix_scan_GBps"]
        sel["frac"] = sel["prefix_scan_GBps"] / peak
        sel["note"] = "no ncu DRAM capture found: frac uses the bytes the prefix scan touches"
    out["rooflines"]["k_select"] = sel
    out["rooflines"]["k_expand"] = {"ms_per_wave": ms[2] / w, "bound": "issue (sort network)",
                                    "algorithmic_GBps": ev * (1448 + 56 + 20 * 250) / (ms[2] / 1e3) / 1e9 if ms[2] > 0 else 0.0}
    out["rooflines"]["k_backup"] = {"ms_per_wave": ms[3] / w, "bound": "latency (pointer chase)"}
    if "f16" in kern:
        k16 = kern["f16"]
        b16 = hist_bytes + P * 24 * 2
        g16 = k16["feat_pos"] * b16 / (k16["feat_ms"] / 1e3) / 1e9 if k16["feat_ms"] > 0 else 0.0
        out["rooflines"]["k_leaf_features_f16_nhwc"] = {
            "bound": "hbm", "achieved": g16, "peak": peak, "unit": "GB/s", "frac": g16 / peak,
            "algorithmic_bytes_per_position": b16, "ms_per_launch": k16["feat_ms"] / max(k16["feat_launches"], 1),
            "note": "the format the timed region uses: fp16 NHWC, 24 channels (17,328 B written per position)"}
    out["kernels_ms_per_wave"] = {"select": ms[0] / w, "leaf_features_f32": ms[1] / w, "expand": ms[2] / w, "backup": ms[3] / w}
    return out


# ---- the reference arm: the compiled reference search on the host cores, same GPU network ---------------
def ref_selfplay(actor, dev, steps, warmup, slice_rollouts=80):
    """BASELINE.md config 3b.  T host threads, one reference game + one reference TreeSearchT
    (oracle/_ref: MCTSAI_T::act, 1 search thread, 8 rollouts per batch, puct 1.5, virtual loss 1,
    persistent tree) each; every wave's 8 leaves go to the SAME GPU network through the callback.
    A step = every game advances its search by `slice_rollouts` rollouts (a tenth of a move; ten
    slices accumulate on the persistent root, then the move is played), so moves = rollouts / 800.
    Two ways of feeding the network are timed and the better one is the baseline:
      one_call_per_wave : each thread calls the network with its own 8 leaves (what a lone game thread sees)
      batched           : a collector gathers the waiting threads' leaves into one call of up to 256 rows,
                          as elf::Batcher does for the reference's game threads (broadcast.h:51-141); more
                          game threads than cores, since they block on the network."""
    import queue

    import numpy as np
    import torch

    from tests import oracles

    if not oracles.have_ref(BOARD):
        return {"unavailable": "oracle/_ref not built"}
    cores = effective_cores()
    P1 = BOARD * BOARD + 1
    lock = threading.Lock()

    tls = threading.local()

    def net(feats):  # feats: float32 numpy [m,18,N,N] -> pi [m,P1], v [m]; pads to a power of two (static shapes)
        m = feats.shape[0]
        mp = 8
        while mp < m:
            mp *= 2
        bufs = getattr(tls, "bufs", None)
        if bufs is None:
            bufs = tls.bufs = {}
        x = bufs.get(mp)
        if x is None:  # one pinned staging buffer per thread and padded size (a pinned allocation per call would
            x = bufs[mp] = torch.zeros((mp, 18, BOARD, BOARD), dtype=torch.float32, pin_memory=dev.type == "cuda")  # handicap this arm)
        x[:m] = torch.from_numpy(feats)
        with lock, torch.no_grad():
            out = actor({"s": x.to(dev, non_blocking=True)})
            pi, v = out["pi"][:m].float().cpu().numpy(), out["V"].reshape(-1)[:m].float().cpu().numpy()
        return pi, v

    results = {}
    for mode, T in (("one_call_per_wave", cores), ("batched", min(8 * cores, 256))):
        evals = [0] * T
        q = queue.Queue()
        stop = threading.Event()

        def collector():
            while not stop.is_set():
                try:
                    first = q.get(timeout=0.05)
                except queue.Empty:
                    continue
                items, rows = [first], first[0].shape[0]
                while rows < NN_BATCH:
                    try:
                        it = q.get_nowait()
                    except queue.Empty:
                        break
                    items.append(it)
                    rows += it[0].shape[0]
                pi, v = net(np.concatenate([it[0] for it in items]))
                o = 0
                for f, box, ev in items:
                    k = f.shape[0]
                    box.append((pi[o:o + k], v[o:o + k]))
                    o += k
                    ev.set()

        start, done = threading.Barrier(T + 1), threading.Barrier(T + 1)
        nsteps = warmup + steps

        def work(tid):
            def cb(feats, hashes):
                evals[tid] += len(hashes)
                if mode == "one_call_per_wave":
                    return net(np.ascontiguousarray(feats))
                box, ev = [], threading.Event()
                q.put((np.array(feats, copy=True), box, ev))
                ev.wait()
                return box[0]

            rng = np.random.default_rng(1000 + tid)
            st = oracles.Ref(BOARD)
            for _ in range(16):
                st.forward(int(rng.choice(np.flatnonzero(st.legal()))))
            m = oracles.RefMcts(BOARD, num_rollouts=slice_rollouts, num_rollouts_per_batch=PER_BATCH, virtual_loss=1,
                                persistent_tree=1, c_puct=1.5, seed=tid, callback=cb)
            slices = 0
            for _ in range(nsteps):
                start.wait()
                r = m.act(st)
                slices += 1
                if slices * slice_rollouts >= ROLLOUTS:  # (80 divides both 800 and 400)
                    if not st.terminated():
                        st.forward(r["best_action"])
                    slices = 0
                done.wait()

        th = [threading.Thread(target=work, args=(i,), daemon=True) for i in range(T)]
        col = threading.Thread(target=collector, daemon=True)
        [t.start() for t in th]
        col.start()
        tot, ev0 = 0.0, 0
        for s in range(nsteps):
            if s == warmup:
                ev0 = sum(evals)
            t0 = time.perf_counter()
            start.wait()
            done.wait()
            if s >= warmup:
                tot += time.perf_counter() - t0
        stop.set()
        [t.join() for t in th]
        col.join()
        moves = steps * T * slice_rollouts / ROLLOUTS
        results[mode] = {"value": moves / tot, "unit": "moves/s", "game_threads": T, "ms_per_step": 1e3 * tot / steps,
                         "nn_positions_per_s": (sum(evals) - ev0) / tot}
    best = max(results, key=lambda k: results[k]["value"])
    return {"value": results[best]["value"], "unit": "moves/s", "cores": cores, "kind": "reference", "mode": best,
            "modes": results, "ms_per_step": results[best]["ms_per_step"],
            "sample": (f"reference TreeSearchT (oracle/_ref), {steps} steps x {results[best]['game_threads']} game threads x "
                       f"{slice_rollouts} rollouts (= {slice_rollouts / ROLLOUTS:.2f} move each) on {cores} host cores, "
                       f"driving the same GPU network; better of {list(results)}")}


def ref_selfplay_fake_net(seconds):
    """BASELINE.md config 3a: the reference TreeSearchT with the shim's deterministic fake net (no network
    cost at all) on every host core, one game per thread: the engine-only rate of the CPU search"""
    from tests import oracles

    if not oracles.have_ref(BOARD):
        return {"unavailable": "oracle/_ref not built"}
    cores = effective_cores()
    done = [0] * cores
    t0 = time.perf_counter()
    deadline = t0 + seconds

    def work(tid):
        st = oracles.Ref(BOARD)
        m = oracles.RefMcts(BOARD, num_rollouts=ROLLOUTS, num_rollouts_per_batch=PER_BATCH, virtual_loss=1,
                            persistent_tree=1, c_puct=1.5, seed=tid)
        while time.perf_counter() < deadline and not st.terminated():
            r = m.act(st)
            st.forward(r["best_action"])
            done[tid] += 1

    th = [threading.Thread(target=work, args=(i,)) for i in range(cores)]
    [t.start() for t in th]
    [t.join() for t in th]
    dt = time.perf_counter() - t0
    return {"value": sum(done) / dt, "unit": "moves/s", "cores": cores, "kind": "reference",
            "sample": f"reference TreeSearchT, {ROLLOUTS} rollouts/move, 1 search thread per game, fake net (no NN cost): "
                      f"{sum(done)} moves in {dt:.1f} s on {cores} threads"}


def run_reference_selfplay(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch

    from elf_b200.model import FusedActor

    if not torch.cuda.is_available():
        emit({"impl": "reference", "unavailable": "config 3b drives the GPU network from the reference search: no CUDA device here"})
        return 0
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    _, net_desc, model = make_network(args, dev)
    actor = FusedActor(model, batchsize=args.nn_batch, dtype=torch.float16, cuda_graph=True)
    cb = ref_selfplay(actor, dev, steps=args.steps, warmup=max(1, args.warmup))
    if "unavailable" in cb:
        emit({"impl": "reference", "unavailable": cb["unavailable"]})
        return 0
    world = args.gpus
    line = {
        "impl": "reference", "metric": "self-play moves/sec (MCTS, 19x19)", "value": cb["value"], "unit": "moves/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 search statistics / fp16 network", "data": "synthetic",
        "config": selfplay_config(args, world, net_desc),
        "reference_arm": ("the reference cannot hold 4096 games: it keeps as many games in flight as its host threads can drive "
                          "(cpu_baseline.modes.*.game_threads) on the same per-move search; a step = every game thread advances its "
                          "search by 80 rollouts (0.1 move); moves/s counts completed rollouts / 800"),
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0

_REAL_STDOUT = None


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else any library prints (e.g. the
    'NCCL version' banner) was re-routed to stderr in main()"""
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT, BOARD
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)  # fd 1 -> stderr for native libraries and stray prints
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 20 for selfplay, 30 for playout)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="selfplay", choices=["selfplay", "playout"])
    ap.add_argument("--games", type=int, default=GAMES_PER_GPU,
                    help="selfplay: games in TOTAL over all GPUs (4096); playout: games per GPU")
    ap.add_argument("--board", type=int, default=19, choices=[9, 19])
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--cpu-steps", type=int, default=6, help="steps of the reference search in our line's cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-board-step", action="store_true")
    ap.add_argument("--plies-per-slot", type=int, default=512)
    ap.add_argument("--playout-layout", type=int, default=-1, choices=[-1, 0, 1],
                    help="playout kernel: 0 = one board row per lane, 1 = two rows per lane (19x19, three games per warp), "
                         "-1 = the library's choice (two rows per lane from 12,288 19x19 games up)")
    ap.add_argument("--parts", type=int, default=2, help="selfplay: half batches interleaved per GPU")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--opening-plies", type=int, default=16, help="random plies every game has played when the search starts")
    ap.add_argument("--blocks", type=int, default=20)
    ap.add_argument("--dim", type=int, default=256)
    ap.add_argument("--nn-batch", type=int, default=NN_BATCH)
    ap.add_argument("--fake-net", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32/float64, "
                         "at most 64 MB; same arguments, same inputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the outputs of --impl ours")
    if args.steps is None:
        args.steps = 30 if args.workload == "playout" else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    BOARD = args.board
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.workload == "playout":
        return run_reference_playout(args) if args.impl == "reference" else run_playout(args)
    global ROLLOUTS
    if BOARD == 9:  # BASELINE configs[4]: 9x9, 16384 concurrent games, 400 rollouts per move
        ROLLOUTS = 400
        if args.games == GAMES_PER_GPU:
            args.games = 16384
    return run_reference_selfplay(args) if args.impl == "reference" else run_selfplay(args)


if __name__ == "__main__":
    sys.exit(main())
