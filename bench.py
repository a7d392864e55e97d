#!/usr/bin/env python
"""bench.py — headline benchmark of the KnightVision B200 hot path (contract: see the task / DESIGN.md §measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload mcts|perft] [--impl ours|reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1; RANK/LOCAL_RANK/WORLD_SIZE from the env).  Rank 0 prints ONE JSON line.
Workloads:
  perft  BASELINE.json configs[1]: perft over 65 536 boards per launch (start position + the reference's six test
         positions, tiled), depth 3.  metric = perft leaf nodes/s.
  mcts   BASELINE.json configs[2]: 4 096 concurrent games per GPU, PUCT self-play with the reference net (default).
  train  BASELINE.json configs[4]: the training step of the learn loop on the 20 x 256 tower (bench_train.py).
  learn  BASELINE.json configs[4]: whole loop iterations, self-play feeding training (bench_learn.py).
`--impl reference` times the CPU implementation of the same path (the oracle port, all host cores) on a bounded
sample of the same workload.
`--dump-outputs DIR` (mcts) writes what the timed window's last move left a caller as DIR/<name>.npy, so that two builds
can be compared output for output on identical (seeded) inputs; see bench_mcts.collect_outputs (rank 0's games only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

PERFT_BOARDS = 65536
PERFT_DEPTH = 3


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class Clocks:
    """nvidia-smi clock / throttle-reason sampler running DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


def _ncu_perft_issue():
    """Issue-slot utilisation and traffic of the perft leaf kernel from the committed ncu capture (profiles/), or None."""
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_perft*.txt")))
    if not files:
        return None
    txt = open(files[-1]).read()
    iss = [float(x) for x in re.findall(r"smsp__issue_active\.avg\.pct_of_peak_sustained_active\s+([0-9.]+)", txt)]
    rd = [float(x) for x in re.findall(r"dram__bytes_read\.sum\s+([0-9.]+) Mbyte", txt)]
    if not iss:
        return None
    return {"issue_active_pct_of_peak": sum(iss) / len(iss), "dram_read_mbyte_per_launch": (sum(rd) / len(rd)) if rd else None,
            "source": os.path.relpath(files[-1], ROOT)}


def perft_roots(n):
    from knightvision_b200 import layout as L
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "perft.json")))
    base = np.array([L.start_line()] + [gold[k]["line"] for k in gold if k != "startpos"], dtype=np.uint64)
    return base[np.arange(n) % len(base)]


# ----------------------------------------------------------------------------------------------------------
def cpu_perft_worker(args):
    from oracle import kv_oracle as O
    lines, depth = args
    tot = 0
    for l in lines:
        tot += int(O.perft2(l, depth)[0])
    return tot


def cpu_perft_throughput(n_boards, depth, procs):
    """Oracle port (oracle/kv_oracle.c) on `procs` host processes over the first n_boards of the workload."""
    import multiprocessing as mp
    from oracle import kv_oracle as O
    O.build()
    roots = perft_roots(n_boards)
    parts = [roots[i::procs] for i in range(procs)]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        tot = sum(pool.map(cpu_perft_worker, [(p, depth) for p in parts]))
    dt = time.perf_counter() - t0
    return tot / dt, tot, dt


def run_reference(args, rank, world):
    """CPU arm: the reference algorithm (oracle port; the Python reference cannot travel to the GPU box)."""
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    if args.workload == "perft":
        # bounded sample: size so that one step is ~2-4 s of all-core CPU work
        n = 64 * procs
        vals = []
        for _ in range(args.warmup if args.warmup < 1 else 1):
            cpu_perft_throughput(n, PERFT_DEPTH, procs)
        t_tot, nodes_tot = 0.0, 0
        for _ in range(args.steps):
            v, nodes, dt = cpu_perft_throughput(n, PERFT_DEPTH, procs)
            vals.append(v); t_tot += dt; nodes_tot += nodes
        value = nodes_tot / t_tot
        line = {"impl": "reference", "metric": "perft_leaf_nodes_per_s", "value": value, "unit": "nodes/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": f"perft depth {PERFT_DEPTH}, start position + the reference's six test positions tiled",
                           "boards_per_step": n},
                "cpu_baseline": {"value": value, "unit": "nodes/s", "cores": procs, "kind": "port",
                                 "sample": f"{n} root boards per step, depth {PERFT_DEPTH}, oracle/kv_oracle.c on {procs} processes"},
                "e2e": {"value": value, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return
    if args.workload == "train":
        import bench_train
        bench_train.run_reference(args)
        return
    import bench_mcts
    bench_mcts.run_reference(args)


# ----------------------------------------------------------------------------------------------------------
def perft_record(args, eng, rank, world, steps, cpu=True):
    """BASELINE configs[1]: perft depth 3 over 65 536 boards per launch and GPU (counts-only leaves), plus the
    start-position depth-5 check (4 865 721, the reference's own count).  Returns the record on rank 0 (None elsewhere)."""
    import torch
    import torch.distributed as dist
    from knightvision_b200 import layout as L
    from knightvision_b200.engine import lines_to_device

    dev = eng.device
    roots_h = perft_roots(PERFT_BOARDS)
    roots = lines_to_device(roots_h, dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.int32, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        # counts-only mode (negative chunk): nodes + category counts, leaves bulk-counted; the order digest is
        # exercised by the parity tests (tests/test_gpu_rules.py), not timed here
        return eng.perft(roots, PERFT_DEPTH, chunk=-PERFT_BOARDS)

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = step()
    torch.cuda.synchronize()
    nodes_per_step = int(out[:, 0].sum().item())
    calls_per_step = int(out[:, 6].sum().item())
    d5 = int(eng.perft_host(L.start_line()[None], 5)[0][0])          # parity spot check inside the bench run
    clocks = Clocks(eng.index)
    clocks.start()
    eng.profile(True)
    eng.profile_read()
    l0 = eng.launches
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.fill_(1)   # flush L2 between timed iterations (outside the timed events)
        a.record()
        step()
        b.record()
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    prof = eng.profile_read()
    eng.profile(False)
    launches = eng.launches - l0
    # e2e: host roots -> C-ABI host entry point -> host results, copies inside the timed region
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = eng.perft_host(roots_h, PERFT_DEPTH, chunk=-PERFT_BOARDS)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()
    assert int(res[:, 0].sum()) == nodes_per_step

    t = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    lvl = eng.perft(roots, PERFT_DEPTH - 1, chunk=-PERFT_BOARDS)      # boards the leaf level visits = perft(d-1) nodes
    torch.cuda.synchronize()
    del flush
    if rank != 0:
        return None
    peaks = measured_peaks()
    leaf_ms, leaf_n = prof["perft_leaf"]
    value = world * nodes_per_step * steps / (dev_ms * 1e-3)
    leaf_boards_per_step = int(lvl[:, 0].sum().item())
    alg_bytes = leaf_boards_per_step * steps * 128.0
    achieved = alg_bytes / (leaf_ms * 1e-3) / 1e9 if leaf_ms > 0 else 0.0
    cpu_rec = None
    if cpu:
        cpu_procs = os.cpu_count() or 1
        cpu_val, cpu_nodes, cpu_dt = cpu_perft_throughput(64 * cpu_procs, PERFT_DEPTH, cpu_procs)
        cpu_rec = {"value": cpu_val, "unit": "nodes/s", "cores": cpu_procs, "kind": "port",
                   "sample": f"{64 * cpu_procs} root boards, depth {PERFT_DEPTH}, oracle/kv_oracle.c on {cpu_procs} processes ({cpu_dt:.1f} s)"}
    return {
        "metric": "perft_leaf_nodes_per_s", "value": value, "unit": "nodes/s", "n_gpus": world,
        "steps": steps, "warmup": warm, "ms_per_step": dev_ms / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": f"perft depth {PERFT_DEPTH} over {PERFT_BOARDS} boards per GPU per launch "
                               "(start position + the reference's six test positions, tiled)",
                   "boards_per_launch": PERFT_BOARDS, "l2": "flushed between timed iterations (256 MB fill)",
                   "movegen_calls_per_step": calls_per_step, "leaf_nodes_per_step": nodes_per_step},
        "parity": {"startpos_depth5": d5, "expected": 4865721, "ok": d5 == 4865721},
        "movegen_calls_per_s": world * calls_per_step * steps / (dev_ms * 1e-3),
        "clocks": clk, "gpu_launches": launches,
        "e2e": {"value": world * nodes_per_step * steps / (e2e_ms * 1e-3), "unit": "nodes/s",
                "h2d_bytes_per_step": PERFT_BOARDS * 128, "d2h_bytes_per_step": PERFT_BOARDS * 64},
        "roofline": {"kernel": "perft_level_kernel<LEAF>", "bound": "hbm", "achieved": achieved, "peak": peaks["hbm"],
                     "unit": "GB/s", "frac": achieved / peaks["hbm"], "traffic": None, "peak_source": peaks["source"],
                     "kernel_ms_per_step": leaf_ms / steps, "kernel_share_of_step": leaf_ms / dev_ms,
                     "issue_slots": _ncu_perft_issue(),
                     "note": "integer/bit kernel: 128 B algorithmic bytes per board visited, so the HBM fraction is tiny by "
                             "construction; what bounds it is instruction issue (issue_slots, from the committed ncu capture)"},
        "kernels_ms_per_step": {k: v[0] / steps for k, v in prof.items() if v[1]},
        "cpu_baseline": cpu_rec,
    }


RULES_BOARDS = int(os.getenv("KV_BENCH_RULES_BOARDS", str(1 << 20)))


def rules_record(args, eng, rank, world, steps):
    """movegen_kernel (getValidMoves) and make_moves_kernel (makeMove) on their own: 2^20 random-playout positions per GPU
    (134 MB of board lines + 537 MB of move lists: larger than the 126 MB L2), achieved GB/s against the measured HBM peak.
    Algorithmic bytes (DESIGN.md section 4): movegen 128 B line read + 2 B x moves + 8 B counts/flags per board; make-move
    128 B read + 128 B write + 2 B move word."""
    import torch
    import torch.distributed as dist
    dev = eng.device
    n = RULES_BOARDS
    lines = eng.random_positions(n, 40, 4242 + rank)
    moves = torch.empty((n, 256), dtype=torch.int16, device=dev)
    counts = torch.empty(n, dtype=torch.int32, device=dev)
    flags = torch.empty(n, dtype=torch.int32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(3):
        eng.movegen(lines, moves, counts, flags)
    torch.cuda.synchronize()
    avg_moves = float(counts.float().mean().item())
    pick = moves[:, 0].contiguous()                     # first legal move of every board (0xFFFF-safe: counts > 0 by construction)
    pick = torch.where(counts > 0, pick, torch.full_like(pick, -1))
    work = lines.clone()
    for _ in range(2):
        work.copy_(lines)
        eng.make_moves(work, pick)
    eng.profile(True)
    eng.profile_read()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        eng.movegen(lines, moves, counts, flags)
    b.record()
    barrier()
    mg_ms = a.elapsed_time(b)
    mm_ms = 0.0
    for _ in range(steps):
        work.copy_(lines)
        torch.cuda.synchronize()
        a.record()
        eng.make_moves(work, pick)
        b.record()
        torch.cuda.synchronize()
        mm_ms += a.elapsed_time(b)
    prof = eng.profile_read()
    eng.profile(False)
    t = torch.tensor([mg_ms, mm_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    mg_ms, mm_ms = float(t[0]), float(t[1])
    del moves, work
    if rank != 0:
        return None
    peaks = measured_peaks()
    mg_bytes = n * (128 + 2 * avg_moves + 8) * steps
    mm_bytes = n * (128 + 128 + 2) * steps
    mg_gbs = mg_bytes / (mg_ms * 1e-3) / 1e9
    mm_gbs = mm_bytes / (mm_ms * 1e-3) / 1e9
    ncu = _ncu_rules()
    return {
        "metric": "movegen_boards_per_s", "value": world * n * steps / (mg_ms * 1e-3), "unit": "boards/s", "n_gpus": world,
        "steps": steps, "higher_is_better": True, "dtype": "u64", "data": "synthetic",
        "config": {"workload": f"{n} boards per GPU (k in [0,40) random legal plies from the initial position), "
                               "kv_movegen over all of them per step; kv_make_moves plays the first legal move of each",
                   "avg_legal_moves": avg_moves, "l2": "board lines + move lists (671 MB) exceed the 126 MB L2"},
        "ms_per_step": mg_ms / steps,
        "roofline": {"kernel": "movegen_kernel (8 lanes per board, four boards per warp)", "bound": "hbm", "achieved": mg_gbs, "peak": peaks["hbm"],
                     "unit": "GB/s", "frac": mg_gbs / peaks["hbm"], "traffic": (ncu or {}).get("movegen_dram_bytes"),
                     "peak_source": peaks["source"], "issue_active_pct": (ncu or {}).get("movegen_issue_pct"),
                     "ncu_source": (ncu or {}).get("source"),
                     "note": "integer/bit kernel: issue-bound, not HBM-bound — the achieved GB/s is reported because north_star "
                             "asks for it; the issue-slot figure (committed ncu capture) is what bounds it"},
        "make_moves": {"value": world * n * steps / (mm_ms * 1e-3), "unit": "boards/s", "ms_per_step": mm_ms / steps,
                       "roofline": {"kernel": "make_moves_kernel", "bound": "hbm", "achieved": mm_gbs, "peak": peaks["hbm"],
                                    "unit": "GB/s", "frac": mm_gbs / peaks["hbm"],
                                    "traffic": (ncu or {}).get("make_moves_dram_bytes"),
                                    "issue_active_pct": (ncu or {}).get("make_moves_issue_pct")}},
        "kernels_ms_per_step": {k: v[0] / steps for k, v in prof.items() if v[1]},
    }


def _ncu_rules():
    """Issue-slot utilisation and DRAM bytes per launch of movegen_kernel / make_moves_kernel from the committed capture."""
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_rules_kernels*.txt")))
    if not files:
        return None
    out = {"source": os.path.relpath(files[-1], ROOT)}
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    txt = open(files[-1]).read()
    for key, name in (("movegen", "movegen_kernel"), ("make_moves", "make_moves_kernel")):
        m = re.search(r"== " + name + r"[^\n]*\n(.*?)(?=\n== |\Z)", txt, re.S)
        if not m:
            continue
        blk = m.group(1)
        iss = re.search(r"smsp__issue_active\.avg\.pct_of_peak_sustained_active\s+([0-9.]+)", blk)
        rd = re.search(r"dram__bytes_read\.sum\s+([0-9.]+) (\w*byte)", blk)
        wr = re.search(r"dram__bytes_write\.sum\s+([0-9.]+) (\w*byte)", blk)
        if iss:
            out[key + "_issue_pct"] = float(iss.group(1))
        if rd and wr:
            out[key + "_dram_bytes"] = float(rd.group(1)) * unit[rd.group(2)] + float(wr.group(1)) * unit[wr.group(2)]
    return out


def run_perft(args, rank, world, local_rank):
    from knightvision_b200.engine import Engine
    eng = Engine(local_rank)
    rec = perft_record(args, eng, rank, world, steps=args.steps)
    rules = rules_record(args, eng, rank, world, steps=max(2, min(args.steps, 5)))
    if rank == 0:
        rec["movegen"] = rules
        print(json.dumps(rec), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=["mcts", "perft", "train", "learn"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (mcts workload)")
    args, _ = ap.parse_known_args()
    if args.workload is None:
        args.workload = "mcts" if os.path.exists(os.path.join(ROOT, "bench_mcts.py")) else "perft"
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "ours" or args.workload != "mcts":
            ap.error("--dump-outputs is implemented for the mcts workload of --impl ours")
        try:                        # a directory that cannot be written fails here, before any GPU work
            os.makedirs(args.dump_outputs, exist_ok=True)
        except OSError as e:
            ap.error(f"--dump-outputs: {e}")
        if not os.access(args.dump_outputs, os.W_OK | os.X_OK):
            ap.error(f"--dump-outputs: {args.dump_outputs} is not writable")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: knightvision_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        if args.workload == "perft":
            run_perft(args, rank, world, local_rank)
        elif args.workload == "train":
            import bench_train
            bench_train.run(args, rank, world, local_rank)
        elif args.workload == "learn":
            import bench_learn
            bench_learn.run(args, rank, world, local_rank)
        else:
            import bench_mcts
            bench_mcts.run(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
