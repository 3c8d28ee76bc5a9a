#!/usr/bin/env python3
"""bench.py — env steps/s of the batched connect_four ApplyAction hot path (BASELINE.json configs[1]).

  python bench.py --gpus N --steps K --warmup W          # our arm (CUDA, through the C ABI)
  python bench.py --impl reference --gpus N ...          # the CPU arm on the box's host cores
  python bench.py ... --dump-outputs DIR                  # also write what the last timed step computed, DIR/<name>.npy

One "step" = one pass of State::ApplyAction over one batch of 1,048,576 connect_four states (SoA, 16 B per
state) with one legal action per state.  The (state, action) stream is synthetic: every lane is advanced
k_i ~ U{0..20} uniformly random legal plies from the start (non-terminal), then one uniformly random legal
action is drawn per lane (SURVEY.md §8d config 2).  Every timed step re-applies that action stream to a fresh
private copy of the snapshot (made before the timed region; K+W copies = far more than L2), so all steps do equal
work and none finds its inputs cached.

Printed JSON (one line, rank 0): metric/value = ApplyAction/s with states and actions resident in HBM;
e2e = the same env step through b2s_step_fused_host_compact with pinned HOST buffers (H2D uint8 actions, D2H one
status byte per lane — terminal / outcome / next legal mask — inside the timed region; the float32-returns entry
b2s_step_fused_host is timed as well and reported under extras); roofline = algorithmic bytes / CUDA-event time of
the apply kernel vs the measured HBM peak; cpu_baseline = the CPU arm on a bounded sample.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_STATES = 1 << 20
MAX_PREFIX = 20
BYTES_APPLY = 36          # 16 R state + 4 R action + 16 W state   (SURVEY.md §8d)
BYTES_FUSED = 49          # + 1 W terminal + 8 W returns + 4 W mask
METRIC = "connect_four ApplyAction env steps/sec (batched)"
UNIT = "steps/s"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------ CPU arm

def cpu_arm(n_sample, threads, reps, seed=0x5EED):
    """ApplyAction of the CPU implementation on `threads` host threads over a bounded sample, `reps` passes.
    Returns (steps/s over all passes, kind, per-pass seconds).  kind = "reference" when oracle/_ref holds the
    unmodified reference build (oracle/ref_build.mk), else "port" (the oracle restatement)."""
    ref = os.path.join(ROOT, "oracle", "_ref", "ref_bench")
    if os.path.exists(ref):
        try:
            out = subprocess.run([ref, "apply", "connect_four", str(n_sample), str(MAX_PREFIX), str(seed),
                                  str(threads), str(reps)], capture_output=True, text=True, timeout=900)
            if out.returncode == 0:
                d = json.loads(out.stdout.strip().splitlines()[-1])
                return d["steps_per_s"], "reference", d["per_rep_seconds"]
        except Exception:
            pass
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import OracleGame, lib
    L = lib()
    L.orc_bench_apply.restype = C.c_double
    L.orc_bench_apply.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_uint64, C.c_int, C.c_int,
                                  C.POINTER(C.c_double), C.POINTER(C.c_double)]
    g = OracleGame("connect_four")
    secs = C.c_double()
    per = (C.c_double * reps)()
    v = L.orc_bench_apply(g._g, n_sample, MAX_PREFIX, seed, threads, reps, C.byref(secs), per)
    return v, "port", list(per)


def cpu_loops():
    """The unmodified reference's MCTSBot / CFRSolver / random playouts on the host (bounded samples), when
    oracle/_ref/ref_bench was shipped; reported beside the device numbers in extras."""
    ref = os.path.join(ROOT, "oracle", "_ref", "ref_bench")
    if not os.path.exists(ref):
        return None
    out = {}
    for key, argv in (("mcts_go9x9_1thread", ["mcts", "go(board_size=9)", "2000", "1", "1"]),
                      ("mcts_go9x9_16threads", ["mcts", "go(board_size=9)", "2000", "1", "16"]),
                      ("cfr_leduc", ["cfr", "leduc_poker", "20"]),
                      ("mccfr_external_leduc_1thread", ["mccfr", "leduc_poker", "10000", "1"]),
                      ("rollouts_breakthrough_1thread", ["rollout", "breakthrough", "5000", "1", "1"]),
                      ("rollouts_breakthrough_16threads", ["rollout", "breakthrough", "5000", "1", "16"]),
                      ("rollouts_tic_tac_toe_1thread", ["rollout", "tic_tac_toe", "100000", "1", "1"])):
        try:
            r = subprocess.run([ref] + argv, capture_output=True, text=True, timeout=300)
            out[key] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:          # noqa: BLE001
            out[key] = {"error": str(e)}
    return out


def host_cpus():
    host = os.cpu_count() or 1
    try:
        host = min(host, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return host


def run_reference(args):
    """The unmodified reference's State::ApplyAction on the box's host cores, on OUR arm's configuration: 1,048,576 states
    per step, same U{0..20}-ply stream.  Thread count is fixed and stated (all host CPUs; no per-run calibration); the
    1-thread figure — the reference's native mode — is reported next to it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    host = host_cpus()
    n_sample = N_STATES
    # Fixed thread count, no calibration: 16.  The reference steps one heap-allocated State per lane, so its throughput
    # peaks around 16 threads on these hosts and FALLS beyond (measured on the 128-CPU box: 1 thread 2.7e6/s, 16 threads
    # ~1.1e7/s, all 128 threads 4.5e5/s — allocator and memory contention); 16 gives the reference its best showing, and
    # the 1-thread and all-CPU figures are reported next to it.
    threads = min(16, host)
    _, kind, per = cpu_arm(n_sample, threads, args.warmup + args.steps)
    times = per[args.warmup:]
    ms = 1e3 * sum(times) / max(len(times), 1)
    value = n_sample / (ms / 1e3) if ms > 0 else 0.0
    v1, _, per1 = cpu_arm(n_sample, 1, 4)
    vall, _, perall = cpu_arm(n_sample, host, 3) if host > threads else (value, None, times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "connect_four batched ApplyAction, 1,048,576-state SoA batch per GPU (BASELINE configs[1])",
                   "states_per_step_per_gpu": n_sample, "prefix_plies": "U{0..%d}" % MAX_PREFIX,
                   "cpu_arm": "one heap-allocated open_spiel::State per lane, ApplyAction timed, Clone excluded"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": "%d states per step x %d steps on %d threads (fixed, no calibration) of %d host CPUs" % (n_sample, len(times), threads, host),
                         "host_cores": host, "value_1_thread": v1,
                         "sample_1_thread": "%d states x 4 passes, 1 thread (%.2f s timed)" % (n_sample, sum(per1)),
                         "value_all_cpus": vall, "sample_all_cpus": "%d states x 3 passes on all %d CPUs" % (n_sample, host)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm

class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0:
                    self.samples.append([x.strip() for x in out.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def build_workload(torch, game, n, dev, seed, with_history=False):
    """Snapshot batch of n non-terminal positions + one legal action per lane (all on device).  with_history also returns
    the plies that built every lane, int32 [n, MAX_PREFIX] (-1 = no move), so the exact benched batch can be replayed on the
    reference (tests/test_gpu_bench_workload.py)."""
    snap = game.new_batch(n)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    k = torch.randint(0, MAX_PREFIX + 1, (n,), device=dev, generator=gen)
    cols = torch.arange(7, device=dev, dtype=torch.int32)

    def random_legal(mask_words):
        legal = ((mask_words[:, :1] >> cols) & 1).bool()                       # [n,7]
        score = torch.rand((n, 7), device=dev, generator=gen).masked_fill(~legal, -1.0)
        return score.argmax(dim=1).to(torch.int32), legal.any(dim=1)

    # advance lane i by k_i plies, never stepping INTO a terminal state (keep the pre-terminal position)
    probe = game.new_batch(n)
    hist = []
    for t in range(MAX_PREFIX):
        a, has = random_legal(snap.legal_actions_mask_words())
        a = torch.where((t < k) & has, a, torch.full_like(a, -1))
        probe.copy_from(snap)
        probe.apply_actions(a)
        _, term, _ = probe.status()
        a = torch.where(term.bool(), torch.full_like(a, -1), a)               # do not enter terminal states
        snap.apply_actions(a)
        if with_history:
            hist.append(a.clone())
    actions, has = random_legal(snap.legal_actions_mask_words())
    assert bool(has.all())
    snap.check_errors()
    if with_history:
        return game, snap, actions.contiguous(), torch.stack(hist, dim=1).contiguous()
    return game, snap, actions.contiguous()


def run_gpu(args):
    import torch
    import open_spiel_b200 as b2
    from open_spiel_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the b200 arm has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # NUMA: pin this rank to the CPUs next to its GPU BEFORE any pinned buffer is allocated (first touch), so the
    # host<->device copies of the e2e path do not cross the socket interconnect (GPUs 4-7 hang off node 1).
    numa_cpus = b2.bind_host_to_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    n = N_STATES                      # per GPU: weak scaling, independent shards, no data-path collective
    K, W = args.steps, args.warmup
    game = b2.Game("connect_four", device=local)
    _, snap, actions0 = build_workload(torch, game, n, dev, seed=0x5EED + rank)
    # "Inputs larger than L2": every timed step owns a private copy of the 16 MiB batch and of the 4 MiB action
    # array ((K+W) x 20 MiB in total, far beyond the 126 MB L2), so no step can find its lines cached; in steady
    # state each step reads 20 MiB from HBM and leaves 16 MiB of dirty lines for later eviction — exactly the
    # algorithmic traffic.  Nothing but the K apply launches sits between the two timing events.
    C = min(K, 512)                   # timed launches per graph; larger K runs ceil(K/C) graphs, restoring between
    slots = C + W
    works = [game.new_batch(n) for _ in range(slots)]
    acts = [actions0.clone() for _ in range(slots)]

    def restore():
        for w_ in works:
            w_.copy_from(snap)

    L = _lib.lib()
    stream = torch.cuda.Stream(device=dev)
    sides = [torch.cuda.Stream(device=dev) for _ in range(3)]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def capture(fn_per_slot, lo, hi, n_streams=1):
        """CUDA graph of launches [lo, hi) (the env loop is launch-bound; graphs keep the host out of it).  n_streams > 1:
        step i runs on stream i mod n_streams — the steps work on DIFFERENT batches, so they are independent and the
        graph says so (parallel branches) instead of serialising them on one stream."""
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            if n_streams == 1:
                for i in range(lo, hi):
                    fn_per_slot(i)
            else:
                lanes = [stream] + sides[:n_streams - 1]
                fork = torch.cuda.Event()
                fork.record(stream)
                for sd in lanes[1:]:
                    sd.wait_event(fork)
                for i in range(lo, hi):
                    with torch.cuda.stream(lanes[(i - lo) % n_streams]):
                        fn_per_slot(i)
                for sd in lanes[1:]:
                    join = torch.cuda.Event()
                    join.record(sd)
                    stream.wait_event(join)
        return g

    def time_graphs(fn_per_slot, reps=3, n_streams=1):
        """W warm-up launches, then exactly K timed launches (in graphs of <= C) bracketed by barrier + synchronize;
        returns the best-of-`reps` max-over-ranks milliseconds for the K launches (CUDA events on the launching stream)."""
        restore()
        torch.cuda.synchronize()
        chunks = [(k0, min(C, K - k0)) for k0 in range(0, K, C)]
        gw = capture(fn_per_slot, 0, W, n_streams)
        graphs = {}
        for _, cnt in chunks:
            if cnt not in graphs:
                graphs[cnt] = capture(fn_per_slot, W, W + cnt, n_streams)
        best = None
        for _ in range(reps):
            total = 0.0
            for _, cnt in chunks:
                restore()
                barrier()
                with torch.cuda.stream(stream):
                    gw.replay()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    graphs[cnt].replay()
                    e1.record(stream)
                barrier()
                total += e0.elapsed_time(e1)
            ms = total
            if dist is not None:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            best = ms if best is None else min(best, ms)
        return best

    def maxtime(seconds):
        if dist is None:
            return seconds
        t = torch.tensor([seconds], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    mask = torch.empty((n, 1), dtype=torch.int32, device=dev)
    term = torch.empty((n,), dtype=torch.uint8, device=dev)
    rets = torch.empty((n, 2), dtype=torch.float32, device=dev)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = L.b2s_launch_count()
    # ---- headline: ApplyAction, device-resident.  The K steps work on K different batches, i.e. they are independent, and
    # the graph says so: two parallel chains (step i on chain i mod 2), so that the grid ramp-up of one step overlaps the
    # drain of the previous one.  (The same K steps forced into one chain — every launch ordered after the previous one, as
    # round 1 timed them — and 4 chains are measured right after and reported beside it.)
    ms_apply_total = time_graphs(lambda i: works[i].apply_actions(acts[i]), n_streams=2)
    for w_ in works:
        w_.check_errors()
    outputs = step_outputs(torch, works[W + (K - 1) % C], dev) if args.dump_outputs and rank == 0 else None
    ms_apply_s1 = time_graphs(lambda i: works[i].apply_actions(acts[i]), reps=2, n_streams=1)
    ms_apply_s4 = time_graphs(lambda i: works[i].apply_actions(acts[i]), reps=2, n_streams=4)
    for w_ in works:
        w_.check_errors()
    # ---- extras: fused step, legal mask -------------------------------------------------------------
    ms_fused_total = time_graphs(lambda i: works[i].step(acts[i], mask, term, rets), reps=2)
    ms_mask_total = time_graphs(lambda i: works[i].legal_actions_mask_words(out=mask), reps=2)
    # ---- e2e: host buffers, one synchronous C-ABI call per step (H2D + kernel + D2H + sync inside the call) ----------
    act_h8 = actions0.to(torch.uint8).cpu().pin_memory()         # compact entry: 1 B in, 1 B out per lane
    status_h = torch.empty((n,), dtype=torch.uint8).pin_memory()
    act_h = actions0.cpu().pin_memory()                          # float entry: 4 B in, 13 B out per lane
    mask_h = torch.empty((n, 1), dtype=torch.int32).pin_memory()
    term_h = torch.empty((n,), dtype=torch.uint8).pin_memory()
    rets_h = torch.empty((n, 2), dtype=torch.float32).pin_memory()

    def time_host_calls(call, reps=3):
        """K synchronous host-buffer calls after W warm-up calls, wall clock around them; best of `reps` passes (like the
        device-resident figure), max over ranks."""
        restore()
        for w_ in works:                      # outside the timed region: every batch allocates its staging buffers and captures
            call(w_, n)                       # the pipeline graph for these host buffers (first call on a batch)
        best = None
        for _ in range(reps):
            restore()
            barrier()
            for i in range(W):
                call(works[i], n)
            barrier()
            total = 0.0
            for k0 in range(0, K, C):
                if k0:
                    restore()
                    barrier()
                t0 = time.perf_counter()
                for i in range(W, W + min(C, K - k0)):
                    call(works[i], n)             # returns after the D2H copies completed
                torch.cuda.synchronize()
                total += (time.perf_counter() - t0) * 1e3
            if dist is not None:
                t = torch.tensor([total], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                total = float(t.item())
            barrier()
            best = total if best is None else min(best, total)
        return best

    ms_e2e_total = time_host_calls(lambda w_, m: w_.step_host_compact(act_h8, status_h, n=m))
    status_snapshot = status_h.clone()
    ms_e2e_f32_total = time_host_calls(lambda w_, m: w_.step_host(act_h, mask_h, term_h, rets_h, n=m))
    # the two entry points must describe the same step: terminal flags and legal masks agree lane for lane
    e2e_consistent = bool(((status_snapshot >> 7) == term_h).all()) and \
        bool((torch.where(term_h.bool(), torch.zeros_like(mask_h[:, 0]), mask_h[:, 0]).to(torch.uint8) ==
              torch.where(term_h.bool(), torch.zeros_like(status_snapshot), status_snapshot & 0x7F)).all())
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    for w_ in works:
        w_.check_errors()
    total_launches = L.b2s_launch_count() - launches0
    del works, acts
    torch.cuda.empty_cache()

    # ---- SURVEY §8(d): the same kernel on a batch larger than L2 (64M lanes = 1 GiB of state) ----------------------
    big_n = n * 64
    big = game.new_batch(big_n)
    acts_big = actions0.repeat(64).contiguous()
    big_ms = []
    for rep in range(6):
        for t in range(64):
            big.copy_from(snap, src_begin=0, dst_begin=t * n, count=n)
        barrier()
        with torch.cuda.stream(stream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            big.apply_actions(acts_big)
            e1.record(stream)
        barrier()
        if rep:
            big_ms.append(e0.elapsed_time(e1))
    big.check_errors()
    ms_big = maxtime(sum(big_ms) / len(big_ms))
    del big, acts_big
    torch.cuda.empty_cache()

    # ---- the loops that drive the step kernels (BASELINE configs[2..4]); reported under "extras" -------------
    loops = {}
    from open_spiel_b200 import parallel
    # MCTS: go 9x9, RandomRolloutEvaluator(1), uct_c=2, solve; independent roots sharded over GPUs
    go = b2.Game("go", {"board_size": 9}, device=local)

    def mcts_line(trees, sims, nodes=0):
        roots = go.new_batch(trees)
        b2.mcts_search(roots, 8, seed=1, tree_index_offset=rank * trees, max_nodes_total=nodes)   # warm-up: allocations, table upload
        barrier()
        t0 = time.perf_counter()
        out = b2.mcts_search(roots, sims, uct_c=2.0, n_rollouts=1, solve=True, seed=1, tree_index_offset=rank * trees,
                             max_nodes_total=nodes)
        torch.cuda.synchronize()
        dt = maxtime(time.perf_counter() - t0)
        nsims = parallel.allreduce_stats(out["sims_run"].sum().to(torch.int64).reshape(1))
        res = {"sims_per_s": float(nsims.item()) / dt, "trees_per_gpu": trees, "sims_per_tree": sims, "seconds": dt,
               "errors": roots.error_count()[0], "nodes_used_rank0": b2.mcts_nodes_used(roots)}
        del roots, out
        torch.cuda.empty_cache()
        return res

    loops["mcts_go9x9"] = mcts_line(65536, 128)          # throughput grows with resident trees until ~14 warps/SM (DESIGN.md §4)
    # deep trees (BASELINE configs[2] is 100k sims/move; a full 100k-sim run of enough trees takes minutes and is recorded
    # in profiles/): steady state at 10k simulations per tree, where descents are ~10 levels deep
    loops["mcts_go9x9_deep"] = mcts_line(args.deep_trees, args.deep_sims, nodes=args.deep_trees * 240000)
    # self-play rollouts: breakthrough 8x8, 2^20 games per GPU, statistics all-reduced
    bt = b2.Game("breakthrough", device=local)
    games = 1 << 20
    bb = bt.new_batch(games)
    bb.rollout(seed=9, lane_offset=rank * games, n=1024)
    bb.reset()
    barrier()
    t0 = time.perf_counter()
    rets_r, plies_r = bb.rollout(seed=9, lane_offset=rank * games)
    torch.cuda.synchronize()
    dt = maxtime(time.perf_counter() - t0)
    st = parallel.rollout_stats(rets_r, plies_r).tolist()
    loops["rollouts_breakthrough"] = {"games_per_s": st[4] / dt, "plies_per_s": st[3] / dt, "p0_wins": st[0], "p1_wins": st[1],
                                      "games": st[4], "seconds": dt}
    del bb, rets_r, plies_r
    # CFR: leduc_poker at the configured 100,000 iterations; single-GPU bit-exact solver (replicated per rank) and, for
    # N > 1, the NCCL-sharded solver
    leduc = b2.Game("leduc_poker", device=local)
    solver = b2.CFRSolver(leduc)
    solver.evaluate_and_update_policy(10)
    torch.cuda.synchronize()
    iters = args.cfr_iters
    t0 = time.perf_counter()
    solver.evaluate_and_update_policy(iters)
    torch.cuda.synchronize()
    dt = maxtime(time.perf_counter() - t0)
    loops["cfr_leduc"] = {"iters_per_s": iters / dt, "node_visits_per_s": iters * 2 * 9457 / dt, "iters": iters, "seconds": dt,
                          "exploitability": solver.exploitability()}
    if world > 1:
        dsolver = parallel.DistributedCFRSolver(leduc)
        dsolver.evaluate_and_update_policy(5)
        barrier()
        t0 = time.perf_counter()
        dsolver.evaluate_and_update_policy(200)
        torch.cuda.synchronize()
        dt = maxtime(time.perf_counter() - t0)
        loops["cfr_leduc_nccl_sharded"] = {"iters_per_s": 200 / dt, "world": world, "seconds": dt}
    del solver
    # external-sampling MCCFR: leduc_poker, 16384 traversals per update (replicated per rank, seeds differ)
    mc = b2.ExternalSamplingMCCFRSolver(leduc, seed=11 + rank, traversals_per_update=16384)
    mc.run_iteration(2)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mc.run_iteration(50)
    torch.cuda.synchronize()
    dt = maxtime(time.perf_counter() - t0)
    loops["mccfr_external_leduc"] = {"traversals_per_s": world * 2 * 16384 * 50 / dt, "traversals_per_update": 16384,
                                     "iterations": 50, "seconds": dt, "nash_conv_rank0": mc.nash_conv()}
    del mc
    # self-play trajectory recorder: connect_four, 2^18 episodes per GPU with observations (42 x 2^18 x 126 floats)
    c4 = b2.Game("connect_four", device=local)
    eps = 1 << 18
    tb = c4.new_batch(eps)
    tb.record_trajectories(seed=1, lane_offset=rank * eps)
    tb.reset()
    barrier()
    t0 = time.perf_counter()
    tr = tb.record_trajectories(seed=2, lane_offset=rank * eps)
    torch.cuda.synchronize()
    dt = maxtime(time.perf_counter() - t0)
    nbytes = sum(v.numel() * v.element_size() for v in tr.time_major.values() if v is not None)
    dec = parallel.allreduce_stats(tr.lengths.sum().to(torch.int64).reshape(1))
    loops["trajectories_connect_four"] = {"episodes_per_s": world * eps / dt, "decisions_per_s": float(dec.item()) / dt,
                                          "episodes_per_gpu": eps, "output_gbs_per_gpu": nbytes / dt / 1e9, "seconds": dt}
    del tb, tr
    barrier()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    ms_apply, ms_fused, ms_mask = ms_apply_total / K, ms_fused_total / K, ms_mask_total / K
    ms_e2e, ms_e2e_f32 = ms_e2e_total / K, ms_e2e_f32_total / K
    peak, peak_src = hbm_peak()
    value = world * n / (ms_apply / 1e3)
    ach = BYTES_APPLY * n / (ms_apply / 1e3) / 1e9          # per GPU
    cores = os.cpu_count() or 1
    cpu_v, cpu_kind, cpu_per = cpu_arm(1 << 18, 1, 8)
    cpu_secs = sum(cpu_per)
    traffic, traffic_src = None, None
    for name in ("r02_apply_traffic.json", "r01_apply_traffic.json"):       # ncu --set full capture of this kernel (not measured in-run)
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
                traffic_src = "profiles/" + name + " (ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch; constant, not re-measured by this run)"
                break
            except Exception:
                pass

    def frac(ms):
        return BYTES_APPLY * n / (ms / 1e3) / 1e9 / peak

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_apply, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": "connect_four batched ApplyAction, 1,048,576-state SoA batch per GPU (BASELINE configs[1])",
                   "states_per_step_per_gpu": n, "state_bytes": 16, "action_dtype": "int32",
                   "prefix_plies": "U{0..%d}" % MAX_PREFIX,
                   "l2": "inputs larger than L2: every step has its own 16 MiB batch + 4 MiB actions (%d x 20 MiB)" % slots,
                   "timing": "K launches in one CUDA graph between two events, barrier+sync both sides, best of 3, max over ranks; ms_per_step = elapsed / K",
                   "graph_chains": 2,
                   "graph_chains_note": "the K steps are on K different batches (independent), captured as 2 parallel chains; one chain (each step ordered after the previous) is extras.apply_1_chain_*",
                   "parallelism": "independent shards x%d, no data-path collective" % world,
                   "host_numa_cpus": numa_cpus,
                   # the loops that drive the step kernels (BASELINE configs[2..4]); full records under extras.loops
                   "loops_summary": {"mcts_go9x9_sims_per_s": loops["mcts_go9x9"]["sims_per_s"],
                                     "mcts_go9x9_deep_sims_per_s": loops["mcts_go9x9_deep"]["sims_per_s"],
                                     "mcts_go9x9_deep_config": "%d trees x %d simulations per GPU" % (args.deep_trees, args.deep_sims),
                                     "cfr_leduc_iters_per_s": loops["cfr_leduc"]["iters_per_s"],
                                     "cfr_leduc_iters": loops["cfr_leduc"]["iters"],
                                     "rollouts_breakthrough_games_per_s": loops["rollouts_breakthrough"]["games_per_s"]}},
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "kernel": "k_apply<ConnectFourRules,4>",
                     "bytes_per_step": BYTES_APPLY, "peak_source": peak_src,
                     "frac_1_chain": frac(ms_apply_s1 / K), "frac_4_chains": frac(ms_apply_s4 / K),
                     "frac_64M_lanes": BYTES_APPLY * big_n / (ms_big / 1e3) / 1e9 / peak,
                     "note": "achieved = 36 B x 1,048,576 lanes / (elapsed / K).  1M lanes are 5.7 us of pure transfer per launch: launches "
                             "ordered one after the other on a single chain pay a grid ramp + drain each (frac_1_chain, round 1's figure); "
                             "declared independent — they are: different batches — consecutive launches overlap (frac, frac_4_chains); one "
                             "launch over 64M lanes (> L2) is frac_64M_lanes.  The timed region as a whole pays one ramp-up and one drain "
                             "(~8 us, the same with the timing events as graph nodes: profiles/r02_bench_k20.json), i.e. frac ~0.93 at "
                             "--steps 20 and ~0.998 at --steps 200"},
        "cpu_baseline": {"value": cpu_v, "unit": UNIT, "cores": 1, "kind": cpu_kind,
                         "sample": "%d states x 8 passes, 1 thread, Clone excluded (%.2f s timed)" % (1 << 18, cpu_secs),
                         "host_cores": cores},
        "e2e": {"value": world * n / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": n,
                "ms_per_step": ms_e2e, "timing": "wall clock around K synchronous calls after W warm-up calls, best of 3 passes, max over ranks",
                "host_step_graph_replays": int(L.b2s_host_graph_launches()),
                "call": "b2s_step_fused_host_compact (pinned host uint8 actions in; one status byte per lane out: terminal, outcome, next legal mask)",
                "zero_copy_steps": int(L.b2s_host_zero_copy_steps()),
                "path": "the step kernel reads the action bytes from the pinned host buffer and writes the status bytes back itself over PCIe (no DMA copies)"
                        if L.b2s_host_zero_copy_steps() > 0 else "cudaMemcpyAsync H2D, kernel, cudaMemcpyAsync D2H",
                "consistent_with_float_entry": e2e_consistent},
        "gpu_launches": K,
        "extras": {"apply_1_chain_steps_per_s": world * n / (ms_apply_s1 / K / 1e3), "apply_1_chain_ms": ms_apply_s1 / K,
                   "apply_4_chains_steps_per_s": world * n / (ms_apply_s4 / K / 1e3), "apply_4_chains_ms": ms_apply_s4 / K,
                   "apply_64M_lanes_steps_per_s": world * big_n / (ms_big / 1e3), "apply_64M_lanes_ms": ms_big,
                   "apply_64M_lanes_gbs": BYTES_APPLY * big_n / (ms_big / 1e3) / 1e9,
                   "fused_step_steps_per_s": world * n / (ms_fused / 1e3), "fused_ms": ms_fused,
                   "fused_gbs": BYTES_FUSED * n / (ms_fused / 1e3) / 1e9,
                   "legal_mask_per_s": world * n / (ms_mask / 1e3), "legal_mask_ms": ms_mask,
                   "e2e_float_entry": {"value": world * n / (ms_e2e_f32 / 1e3), "ms_per_step": ms_e2e_f32, "h2d_bytes_per_step": 4 * n,
                                       "d2h_bytes_per_step": 13 * n, "call": "b2s_step_fused_host (int32 actions; mask words, terminal, float32 returns)"},
                   "launches_total_incl_setup": total_launches, "loops": loops, "cpu_reference_loops": cpu_loops()},
        "clocks": sampler.summary() if sampler else None,
    }
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


DUMP_OBS_LANES = 4096


def step_outputs(torch, batch, dev):
    """What a caller of the timed ApplyAction step reads back from the batch it advanced: player to move, terminal flag,
    returns and legal-action mask of every lane, and the observation tensor of a fixed, seeded sample of lanes (all of it
    would be 504 MiB)."""
    cur, term, rets = batch.status()
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x0B5)
    lanes = torch.randperm(batch.n, device=dev, generator=gen)[:DUMP_OBS_LANES].sort().values
    obs = batch.observation_tensor(player=0)[lanes]
    mask = batch.legal_actions_mask_words().to(torch.int64) & 0xFFFFFFFF
    return {"current_player": cur.to(torch.float32), "terminal": term.to(torch.float32), "returns": rets.to(torch.float32),
            "legal_mask_words": mask.to(torch.float64), "observation_lanes": lanes.to(torch.float64),
            "observation_sample": obs.to(torch.float32)}


def dump_outputs(directory, outputs):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--deep-trees", type=int, default=8192, help="trees per GPU of the deep MCTS line")
    ap.add_argument("--deep-sims", type=int, default=10000, help="simulations per tree of the deep MCTS line")
    ap.add_argument("--cfr-iters", type=int, default=100000, help="CFRSolver iterations (BASELINE configs[3]: 100k)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
