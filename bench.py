#!/usr/bin/env python
"""bench.py — matches/sec of the search tick (BASELINE.json metric).

A step = one pass of the hot path (one search tick) over one synthetic player pool.
  value  whole-job lobbies/sec with the pool already resident in HBM; the timed region
         of a step is the tick itself (all its kernels), timed with CUDA events on the
         engine's own stream (mm_tick_stats.device_us); max over ranks.  Between steps
         (untimed) the pool is restored from a device snapshot and L2 is flushed by
         writing a buffer larger than L2.
  e2e    same metric through the C ABI with HOST buffers, every step a NEW batch of players:
         mm_enqueue_packed (pinned host columns: u32 handle + u16 mode|rating = 6 B/player H2D
         inside) + mm_enqueue_rejects + mm_tick_packed (lobby headers + u32 member handles D2H
         inside), wall clock.  `pipelined`: two batches in flight — step k+1's upload
         (mm_enqueue_packed_begin) and step k-1's host copies (mm_set_option "async_results") run
         under step k's ingest + tick; `pipelined_results_only`: only the result copies overlap;
         `sequential`: fully blocking calls;
         `u64_api`: the 17 B/player mm_enqueue + 8 B/player mm_tick entry points, blocking.
  strong (N > 1 only) BASELINE configs[3]: ONE pool of the workload's size, its rating groups
         dealt to the ranks (generic/worker.ex:55-69), device-timed like `value`.
  roofline / cpu_baseline: see DESIGN.md §Measurement.
Launch: `python bench.py --gpus 1 --steps K --warmup W`, or under torchrun for N>1
(one rank per GPU; ranks own disjoint rating groups — no data-path collective).
`--impl reference` times the CPU restatement of the reference loop (oracle/).
`--dump-outputs DIR` writes the results of the last timed tick of `value` as DIR/*.npy (see dump_outputs), so that
two builds can be compared output for output on the same seeded pool.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "microservice-matchmaking_b200"

B_ALG_TICK = 22      # SURVEY §8(d) strict-parity mode: read id 8 + rating 4 + mode 1 + team_size 1, write id 8
B_CONSUMED_TICK = 20  # what the tick really moves per player: bin 2 (twice: histogram + placement, the second time
#                       from L2) + id 8 read, id 8 written; rating/mode -> bin is paid at ingest


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        hi = [x for x in sm if x >= 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(hi) if hi else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_ROWS = 1 << 19  # rows kept per array: 2^19 x (4 + 1 + 2 + 1) float64 columns = 32 MiB in all


def read_device_results(pkg, eng, st):
    """Host copies of what the last mm_tick_device left in HBM: lobby headers and u64 member ids."""
    import types

    import numpy as np
    import torch

    def fetch(ptr, nbytes):
        if nbytes == 0:
            return np.empty(0, np.uint8)
        buf = types.SimpleNamespace(__cuda_array_interface__={
            "shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3})
        return torch.as_tensor(buf, device="cuda").cpu().numpy()

    d_lob, d_mem = eng.results_device()
    return (fetch(d_lob, 8 * st.n_lobbies).view(pkg.engine.LOBBY_DTYPE),
            fetch(d_mem, 8 * st.n_matched).view(np.uint64))


def dump_outputs(out_dir, st, lob, mem):
    """One tick's results as float64 .npy files with exact values: tick_counts (pool_before, n_lobbies, n_matched,
    n_residual, n_dead), lobbies (first_member, n_members, mode, group), member_ids (high and low 32 bits).  An array
    longer than DUMP_ROWS is a fixed seeded sample of its rows; <name>_rows holds their row numbers."""
    import numpy as np

    def rows(n):
        if n <= DUMP_ROWS:
            return np.arange(n)
        return np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))

    r_lob, r_mem = rows(len(lob)), rows(len(mem))
    sl, sm = lob[r_lob], mem[r_mem]
    arrays = {
        "tick_counts": np.array([st.pool_before, st.n_lobbies, st.n_matched, st.n_residual, st.n_dead], np.float64),
        "lobbies": np.stack([sl["first_member"], sl["n_members"], sl["mode"], sl["group"]], axis=1).astype(np.float64),
        "lobbies_rows": r_lob.astype(np.float64),
        "member_ids": np.stack([sm >> np.uint64(32), sm & np.uint64(0xFFFFFFFF)], axis=1).astype(np.float64),
        "member_ids_rows": r_mem.astype(np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args, rank, world):
    """--impl reference: the CPU restatement of the reference loop on the host cores."""
    if rank != 0:
        return
    pkg = importlib.import_module(PKG)
    orc = importlib.import_module("oracle.oracle")
    orc.build()
    order = pkg.abi.MM_ORDER_RATING if args.order == "rating" else pkg.abi.MM_ORDER_ARRIVAL
    w = pkg.synth.WORKLOADS[args.workload]
    cfg, mode_idx = pkg.synth.workload_config(args.workload, order, 1, single_mode=not getattr(args, "two_modes", False))
    n = min(w["n"], args.ref_sample)
    ids, rating, mode, _ = pkg.synth.gen_pool(1, n, mode=mode_idx)
    threads = max(1, min(os.cpu_count() or 1, cfg.n_groups))
    for _ in range(args.warmup):
        orc.time_literal(cfg, ids, rating, mode, threads)
    secs, lobbies = 0.0, 0
    for _ in range(args.steps):
        s, nl = orc.time_literal(cfg, ids, rating, mode, threads)
        secs += s; lobbies += nl
    value = lobbies / secs
    sample = f"{n} of {w['n']} players of {args.workload}, literal consume/5 loop, one worker per rating group"
    line = {
        "impl": "reference", "metric": "matches/sec", "value": value, "unit": "lobbies/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32/u64", "data": "synthetic",
        "config": {"workload": args.workload, "order": args.order, "players_per_step": n,
                   "note": "reference BEAM pipeline cannot run here (no Elixir/RabbitMQ, strategist absent): "
                           "CPU restatement oracle/mm_oracle.c, policy S0"},
        "cpu_baseline": {"value": value, "unit": "lobbies/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "lobbies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def stream_leg(pkg, device, seconds, rate, dt_ms, groups=32, max_spread=-1):
    """BASELINE configs[4] on one GPU: Poisson arrivals at `rate` players/s into the resident pool through
    mm_enqueue_packed, one search tick (mm_tick_packed, host results) every dt_ms, real time (the loop is paced with
    the wall clock).  latency = t(host holds the lobby that contains the player) - t(player arrived)."""
    import numpy as np
    abi = pkg.abi
    dt = dt_ms * 1e-3
    n_total = int(rate * seconds)
    rng = np.random.default_rng(1)
    arrive = np.cumsum(rng.exponential(1.0 / rate, n_total))
    _, rating, _, _ = pkg.synth.gen_pool(3, n_total)
    keys = pkg.Engine.pack_key(rating, np.zeros(n_total, np.uint8))
    handles = np.arange(n_total, dtype=np.uint32)  # the host's dense handle = arrival index
    cfg = pkg.synth.make_config(n_groups=groups, modes=(("5v5", 2, 5),), order=abi.MM_ORDER_RATING, capacity=1 << 20,
                                active_capacity=n_total + 1024, device=device)
    cfg.flags |= abi.MM_F_DENSE_IDS
    eng = pkg.Engine(cfg)
    eng.set_option("max_spread", max_spread)
    eng.enqueue_packed(handles[:10], keys[:10]); eng.tick_packed(want_emit_seq=False); eng.remove_packed(handles[:10])  # warm-up
    matched_at = np.full(n_total, np.nan)
    lo, overruns, tick_us, call_us = 10, 0, [], []
    n_ticks = int(seconds / dt)
    t0 = time.perf_counter()
    for k in range(1, n_ticks + 1):
        deadline = t0 + k * dt
        while time.perf_counter() < deadline:
            pass
        now = time.perf_counter() - t0
        hi = int(np.searchsorted(arrive, now))  # everyone who has arrived by now
        if hi > lo:
            eng.enqueue_packed(handles[lo:hi], keys[lo:hi])
        lob, mem, _, st = eng.tick_packed(want_emit_seq=False)
        done = time.perf_counter() - t0
        matched_at[mem] = done
        tick_us.append(st.device_us); call_us.append((done - now) * 1e6)
        overruns += done > (k + 1) * dt
        lo = max(lo, hi)
    eng.close()
    lat = (matched_at - arrive)[10:lo]
    ok = ~np.isnan(lat)
    q = lambda p: float(np.percentile(lat[ok], p) * 1e3)
    return {"workload": "Poisson arrivals into the resident pool, 5v5, %d rating groups, one tick per period" % groups,
            "rate_per_s": rate, "dt_ms": dt_ms, "seconds": seconds, "max_spread": max_spread,
            "players_enqueued": int(lo - 10), "matched": int(ok.sum()), "still_queued": int((~ok).sum()),
            "latency_ms": {"p50": q(50), "p99": q(99), "p99.9": q(99.9), "max": q(100)},
            "tick_device_us": {"mean": float(np.mean(tick_us)), "p99": float(np.percentile(tick_us, 99))},
            "enqueue_plus_tick_call_us": {"mean": float(np.mean(call_us)), "p99": float(np.percentile(call_us, 99))},
            "ticks": n_ticks, "overrun_ticks": int(overruns),
            "note": "strict parity has no time-expanded window (SURVEY F3): a player waits for L-1 more players of its "
                    "(mode, group) and the next tick; the pool holds < L players per partition between ticks"}


def main():
    sys.dont_write_bytecode = True  # the tree may be read-only: bench.py writes nothing there
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config3_10m_g32_5v5")
    ap.add_argument("--order", default="rating", choices=["rating", "arrival"])
    ap.add_argument("--rank-impl", type=int, default=None)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--ref-sample", type=int, default=10_000_000)
    ap.add_argument("--cpu-sample", type=int, default=10_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="under torchrun: skip the configs[3] strong-scaling leg")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--boundary-w", type=int, default=2,
                    help="under torchrun: window of the boundary-pass extension leg (0 = skip)")
    ap.add_argument("--boundary-players", type=int, default=12_000, help="pool size of the boundary-pass leg (sparse: windows fail, residuals sit near the boundaries)")
    ap.add_argument("--stream-seconds", type=float, default=1.0, help="length of the streaming leg (configs[4]); 0 = skip")
    ap.add_argument("--stream-rate", type=float, default=1e6)
    ap.add_argument("--stream-dt-ms", type=float, default=1.0)
    ap.add_argument("--two-modes", action="store_true", help="configure both default modes (1v1, 5v5), not just the workload's")
    ap.add_argument("--tick-impl", type=int, default=None, help="1 = one fused cooperative launch (default), 0 = four launches")
    ap.add_argument("--max-spread", type=int, default=None,
                    help="EXTENSION (policy S1, not the BASELINE workload): a lobby spans at most W rating points")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed tick of `value` returned (rank 0) as "
                         "DIR/<name>.npy, float64, 32 MiB at most")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU tick's results; --impl reference returns none")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import numpy as np
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the search tick has no CPU path "
                         "(use --impl reference for the CPU restatement)")
    torch.cuda.set_device(local)
    import __graft_entry__ as ge
    pkg = ge.build()
    hostutil = importlib.import_module(PKG + ".hostutil")
    numa = {"bound": False} if args.no_numa else hostutil.bind_to_gpu_numa(local)  # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    abi = pkg.abi
    order = abi.MM_ORDER_RATING if args.order == "rating" else abi.MM_ORDER_ARRIVAL
    w = pkg.synth.WORKLOADS[args.workload]
    n, L = w["n"], (2 if w["mode"] == 0 else 10)
    windowed = args.max_spread is not None and args.max_spread >= 0
    cap = n + 65536 + (n if windowed else 0)  # S1 leaves players queued
    cfg, mode_idx = pkg.synth.workload_config(args.workload, order, cap, device=local, single_mode=not args.two_modes)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def options(eng):
        if args.rank_impl is not None:
            eng.set_option("rank_impl", args.rank_impl)
        if args.tick_impl is not None:
            eng.set_option("tick_impl", args.tick_impl)
        if args.max_spread is not None:
            eng.set_option("max_spread", args.max_spread)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def device_timed(cfg_, ids_, rating_, mode_, ts_, steps, warmup, read_results=False):
        """K ticks of one resident pool (restored from a device snapshot, L2 flushed, both untimed); read_results:
        also return host copies of the last tick's lobby headers and member ids (read after the timed region)."""
        eng = pkg.Engine(cfg_)
        options(eng)
        assert eng.enqueue(ids_, rating_, mode_, ts_).all()
        eng.snapshot()

        def one_step():
            eng.restore()
            flush.fill_(1)  # evict the pool from L2
            torch.cuda.synchronize()
            return eng.tick_device()

        for _ in range(warmup):
            st = one_step()
        barrier()
        t0 = time.perf_counter()
        dev_us, phases = [], []
        for _ in range(steps):
            st = one_step()
            dev_us.append(st.device_us)
            phases.append((st.hist_us, st.scan_us, st.place_us, st.epilogue_us))
        barrier()
        wall = time.perf_counter() - t0
        results = read_device_results(pkg, eng, st) if read_results else None
        eng.close()
        return sum(dev_us) * 1e-6, st, phases, wall, results

    # ---- weak leg (the contract's line): every rank holds a full-size pool of its own seed stream -------------
    ids, rating, mode, ts = pkg.synth.gen_pool(1, n, first=rank * n, mode=mode_idx)
    sampler = ClockSampler(local)
    sampler.start()
    tick_s, st, phases, wall_s, last_results = device_timed(cfg, ids, rating, mode, ts, args.steps, args.warmup,
                                                            read_results=bool(args.dump_outputs) and rank == 0)
    launches_per_tick = st.n_launches
    lobbies_per_step = st.n_lobbies
    if world > 1:
        t = torch.tensor([tick_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tick_s = float(t.item())
        tl = torch.tensor([lobbies_per_step, n], device="cuda", dtype=torch.int64)
        dist.all_reduce(tl)
        total_lobbies_per_step, total_players = int(tl[0].item()), int(tl[1].item())
    else:
        total_lobbies_per_step, total_players = lobbies_per_step, n
    value = total_lobbies_per_step * args.steps / tick_s

    # ---- strong leg (BASELINE configs[3]): ONE pool, rating groups dealt to the ranks --------------------------
    strong = None
    if world > 1 and not args.no_strong:
        shard = importlib.import_module(PKG + ".shard")
        g_ids, g_rating, g_mode, g_ts = pkg.synth.gen_pool(1, n, first=0, mode=mode_idx)
        mine = shard.route(cfg, g_rating, world) == rank  # the Generic stage's routing (generic/worker.ex:46-69)
        n_mine = int(mine.sum())
        s_steps = max(3, args.steps // 2)
        s_tick, s_st, s_ph, _, _ = device_timed(cfg, g_ids[mine], g_rating[mine], g_mode[mine], g_ts[mine], s_steps, args.warmup)
        t = torch.tensor([s_tick], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tl = torch.tensor([s_st.n_lobbies, n_mine], device="cuda", dtype=torch.int64)
        tmax = tl.clone(); tmin = tl.clone()
        dist.all_reduce(tl); dist.all_reduce(tmax, op=dist.ReduceOp.MAX); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        s_max = float(t.item())
        strong = {"value": int(tl[0].item()) * s_steps / s_max, "unit": "lobbies/s", "scaling": "strong",
                  "ms_per_step": 1e3 * s_max / s_steps, "steps": s_steps, "players_total": int(tl[1].item()),
                  "players_per_gpu_min": int(tmin[1].item()), "players_per_gpu_max": int(tmax[1].item()),
                  "rating_groups_per_gpu": w["n_groups"] // world, "lobbies_per_step": int(tl[0].item()),
                  "workload": args.workload + f" as ONE pool sharded by rating group over {world} GPUs (BASELINE configs[3]); "
                              "strict parity: no player crosses a group, so no boundary exchange is issued",
                  "timing": "max over ranks of the device-timed ticks (CUDA events on each engine's stream)"}
        # -- EXTENSION leg (not reference behaviour): policy S1 (max_spread W) on the same sharded pool + the boundary
        #    pass: residual players within W of a group boundary owned by another rank travel over NCCL send/recv
        if args.boundary_w > 0:
            Wb, nb_pool = args.boundary_w, min(n, args.boundary_players)
            # a SPARSE slice of the same pool: on the dense 10 M pool every window fills and nobody is left near a boundary
            mine_b = mine[:nb_pool]
            cfg_b, _ = pkg.synth.workload_config(args.workload, abi.MM_ORDER_RATING, int(mine_b.sum()) + 65536, device=local,
                                                 single_mode=not args.two_modes)
            eng = pkg.Engine(cfg_b)
            eng.set_option("max_spread", Wb)
            assert eng.enqueue(g_ids[:nb_pool][mine_b], g_rating[:nb_pool][mine_b], g_mode[:nb_pool][mine_b]).all()
            stb = eng.tick_device()
            comm = shard.DistComm(device=torch.device("cuda", local))
            cache = {}
            barrier()
            t0 = time.perf_counter()
            bp = shard.boundary_pass(pkg, cfg_b, Wb, world, rank, eng, comm, cache=cache)
            barrier()
            bp_ms = 1e3 * (time.perf_counter() - t0)
            for band in cache.values():
                band.close()
            eng.close()
            tb = torch.tensor([bp["sent"], bp["received"], bp["matched"], bp["lobbies"], comm.bytes_sent, stb.n_residual],
                              device="cuda", dtype=torch.int64)
            dist.all_reduce(tb)
            strong["boundary_pass"] = {
                "policy": f"S1 extension, max lobby spread {Wb}", "pool": f"first {nb_pool} players of the workload (sparse)",
                "players_left_queued_by_the_local_ticks": int(tb[5].item()),
                "players_sent_to_the_lower_neighbour": int(tb[0].item()), "players_received": int(tb[1].item()),
                "players_matched_across_a_boundary": int(tb[2].item()), "lobbies": int(tb[3].item()),
                "bytes_over_nccl": int(tb[4].item()), "wall_ms": bp_ms,
                "note": "torch.distributed send/recv on the NCCL process group (NVLink): candidates up, consumed ids back; "
                        "host-orchestrated (pool_read + band engines), so the wall time is dominated by host copies, not "
                        "by the link"}
        del g_ids, g_rating, g_mode, g_ts

    # ---- e2e through the C ABI with host buffers ------------------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        lob_cap, mem_cap = n // L + 8192, n + 65536  # pipelined steps also match the previous step's leftovers
        h_lob = torch.empty(lob_cap, dtype=torch.int64).pin_memory()  # 8-byte mm_lobby_hdr
        S = 2 * args.e2e_steps  # pipelined: the last step's copies are exposed, amortise them over a few more steps

        # -- packed API on a dense-handle engine: 6 B/player up, 4 B/player down
        cfgp, _ = pkg.synth.workload_config(args.workload, order, cap, device=local, single_mode=not args.two_modes)
        cfgp.flags |= abi.MM_F_DENSE_IDS
        cfgp.active_capacity = (S + 4) * n  # handle range: every step brings new players, nobody has left yet
        h_mem32 = torch.empty(mem_cap, dtype=torch.int32).pin_memory()
        h_lob2 = torch.empty(lob_cap, dtype=torch.int64).pin_memory()   # pipelined legs: results alternate between two
        h_mem32b = torch.empty(mem_cap, dtype=torch.int32).pin_memory() # host buffer sets (tick k is read while k+1 runs)
        batches = []
        for k in range(S + 3):
            _, r_k, m_k, _ = pkg.synth.gen_pool(1, n, first=(rank + world * k) * n, mode=mode_idx)
            handles = (np.arange(n, dtype=np.uint64) + np.uint64(k * n)).astype(np.uint32)
            batches.append((pin(handles), pin(pkg.Engine.pack_key(r_k, m_k))))

        def step_packed(eng, b):
            eng.enqueue_packed_raw(n, b[0].data_ptr(), b[1].data_ptr())  # no per-player status transfer ...
            t1 = time.perf_counter()
            rej_idx, _ = eng.enqueue_rejects()                              # ... the nack list comes back instead
            assert len(rej_idx) == 0
            st_ = eng.tick_raw(h_lob.data_ptr(), lob_cap, h_mem32.data_ptr(), mem_cap, packed=True)
            return st_, t1

        eng = pkg.Engine(cfgp); options(eng)
        times, t_enq = [], []
        for it in range(args.e2e_steps + 1):
            barrier()
            t0 = time.perf_counter()
            st2, t1 = step_packed(eng, batches[0])
            dt = time.perf_counter() - t0
            if it:  # first iteration = warm-up
                times.append(dt); t_enq.append(t1 - t0)
            eng.remove_packed(batches[0][0].numpy())  # what the lobby stage does later (game-lobby/worker.ex:80); untimed
        assert st2.n_lobbies == lobbies_per_step
        seq_s, seq_enq_s = sum(times) / len(times), sum(t_enq) / len(t_enq)
        eng.close()
        eng = pkg.Engine(cfgp); options(eng)
        eng.set_option("async_results", 1)
        lob_pipe = 0
        for k in range(S + 1):
            if k == 1:  # batch 0 = warm-up
                eng.results_wait()
                barrier()
                t0 = time.perf_counter()
            st3, _ = step_packed(eng, batches[k + 1])
            if k:
                lob_pipe += st3.n_lobbies
        eng.results_wait()
        res_s = (time.perf_counter() - t0) / S
        eng.close()
        tot_res = lob_pipe / S
        # -- two batches in flight: step k+1's upload (mm_enqueue_packed_begin) runs under step k's ingest, tick and
        #    result copies; every step's host->device and device->host copies are still inside the timed region
        eng = pkg.Engine(cfgp); options(eng)
        eng.set_option("async_results", 1)

        def staged_step(k, last):
            if not last:
                eng.enqueue_packed_begin_raw(n, batches[k + 1][0].data_ptr(), batches[k + 1][1].data_ptr())
            eng.enqueue_packed_end_raw()
            rej_idx, _ = eng.enqueue_rejects()
            assert len(rej_idx) == 0
            hl, hm = (h_lob, h_mem32) if k & 1 else (h_lob2, h_mem32b)
            return eng.tick_raw(hl.data_ptr(), lob_cap, hm.data_ptr(), mem_cap, packed=True).n_lobbies

        # warm-up: two staged steps, so that both staging slots and both result buffer sets exist before the clock starts
        eng.enqueue_packed_begin_raw(n, batches[0][0].data_ptr(), batches[0][1].data_ptr())
        staged_step(0, False)
        staged_step(1, True)
        eng.results_wait()
        barrier()
        lob_pipe = 0
        t0 = time.perf_counter()
        eng.enqueue_packed_begin_raw(n, batches[2][0].data_ptr(), batches[2][1].data_ptr())
        for k in range(2, S + 2):
            lob_pipe += staged_step(k, k == S + 1)
        eng.results_wait()
        e2e_s = (time.perf_counter() - t0) / S
        eng.close()
        del batches
        tot_pipe = lob_pipe / S

        # -- the u64 entry points (17 B/player up, 8 B/player down), blocking: what round 1 measured
        h_ids, h_rating, h_mode, h_ts = pin(ids), pin(rating), pin(mode), pin(ts)
        h_acc = torch.empty(n, dtype=torch.uint8).pin_memory()
        h_mem = torch.empty(mem_cap, dtype=torch.int64).pin_memory()
        eng = pkg.Engine(cfg); options(eng)
        u_times = []
        for it in range(3):
            barrier()
            t0 = time.perf_counter()
            eng.enqueue_raw(n, h_ids.data_ptr(), h_rating.data_ptr(), h_mode.data_ptr(), h_ts.data_ptr(), h_acc.data_ptr())
            st4 = eng.tick_raw(h_lob.data_ptr(), lob_cap, h_mem.data_ptr(), mem_cap)
            if it:
                u_times.append(time.perf_counter() - t0)
            eng.remove(ids)
        eng.close()
        u64_s = sum(u_times) / len(u_times)

        if world > 1:
            t = torch.tensor([e2e_s, seq_s, u64_s, res_s], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s, seq_s, u64_s, res_s = (float(x) for x in t.tolist())
            tl2 = torch.tensor([tot_pipe, tot_res], device="cuda", dtype=torch.float64)
            dist.all_reduce(tl2)
            tot_pipe, tot_res = (float(x) for x in tl2.tolist())
        pipelined = {"value": tot_pipe / e2e_s, "ms_per_step": 1e3 * e2e_s, "steps": S,
                     "call": "per step: mm_enqueue_packed_begin(next step's pinned host handles + keys) + "
                             "mm_enqueue_packed_end(this step's) + mm_enqueue_rejects + mm_tick_packed(host lobbies / "
                             "member handles) with mm_set_option(async_results): two batches in flight — a step's "
                             "upload runs under the previous step's ingest + tick, its device-to-host copies under "
                             "the next step; the first upload and mm_results_wait after the last step are inside "
                             "the timed region"}
        results_only = {"value": tot_res / res_s, "ms_per_step": 1e3 * res_s, "steps": S,
                        "call": "per step: blocking mm_enqueue_packed + mm_enqueue_rejects + mm_tick_packed with "
                                "async_results (only the device-to-host copies overlap the next step)"}
        sequential = {"value": total_lobbies_per_step / seq_s, "ms_per_step": 1e3 * seq_s, "steps": len(times),
                      "enqueue_ms": 1e3 * seq_enq_s, "tick_and_d2h_ms": 1e3 * (seq_s - seq_enq_s),
                      "call": "blocking mm_enqueue_packed + mm_enqueue_rejects + blocking mm_tick_packed, one step at a time"}
        legs = {"pipelined": pipelined, "pipelined_results_only": results_only, "sequential": sequential}
        best_name = max(legs, key=lambda k: legs[k]["value"])  # every leg has all of its copies inside the timed region
        best = legs[best_name]
        e2e = {"value": best["value"], "unit": "lobbies/s",
               "h2d_bytes_per_step": n * (4 + 2), "d2h_bytes_per_step": 8 + st2.n_matched * 4 + st2.n_lobbies * 8,
               "ms_per_step": best["ms_per_step"], "steps": best["steps"], "call": best["call"],
               "mode": best_name,
               "ids": "dense 32-bit host handles (MM_F_DENSE_IDS; the host owns the UUID <-> handle table, SURVEY §7.3)",
               "pipelined": pipelined, "pipelined_results_only": results_only, "sequential": sequential,
               "u64_api": {"value": total_lobbies_per_step / u64_s, "ms_per_step": 1e3 * u64_s,
                           "h2d_bytes_per_step": n * (8 + 4 + 1 + 4), "d2h_bytes_per_step": n + st4.n_matched * 8 + st4.n_lobbies * 8,
                           "call": "blocking mm_enqueue(pinned u64 ids, i32 rating, u8 mode, u32 ts; accepted[] back) + "
                                   "blocking mm_tick(host lobbies / u64 member ids)"},
               "numa": numa}
    stream = None
    if args.stream_seconds > 0 and not args.no_e2e and rank == 0 and world == 1:
        stream = stream_leg(pkg, local, args.stream_seconds, args.stream_rate, args.stream_dt_ms)
    clocks = sampler.stop()  # sampled across the device-timed ticks and the e2e steps

    # ---- CPU baseline (rank 0, N=1 only): the oracle's literal loop on a bounded sample ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        orc = importlib.import_module("oracle.oracle")
        ns = min(n, args.cpu_sample)
        s1, nl1 = orc.time_literal(cfg, ids[:ns], rating[:ns], mode[:ns], 1)
        cpu = {"value": nl1 / s1, "unit": "lobbies/s", "cores": 1, "kind": "port",
               "sample": f"first {ns} of {n} players of {args.workload}; oracle/mm_oracle.c literal consume/5 loop, "
                         f"1 thread, {s1:.2f} s", "players_per_s": ns / s1}

    if rank == 0:
        peak, peak_src = peaks()
        tick_avg_s = tick_s / args.steps
        fused = launches_per_tick == 1
        ach = B_ALG_TICK * n / tick_avg_s / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "tick_traffic.json")
        if os.path.exists(tp) and args.workload == "config3_10m_g32_5v5" and args.order == "rating":
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch" if fused else "dram_bytes_split_launches")
            except Exception:
                pass
        line = {
            "metric": "matches/sec", "value": value, "unit": "lobbies/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tick_s / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32/u64", "data": "synthetic",
            "config": {"workload": args.workload, "players_per_gpu": n, "rating_groups_per_gpu": w["n_groups"],
                       "players_total": total_players,
                       "lobby_size": L, "order": args.order, "ratings": "uniform 0..5000, seed 1",
                       "modes_configured": cfg.n_modes, "launches_per_tick": launches_per_tick,
                       "policy": ("S0 (reference behaviour)" if not windowed else
                                  f"S1 extension: max lobby spread {args.max_spread} rating points"),
                       "players_left_queued_per_step": int(st.n_residual),
                       "parallelism": f"rating-group shards x{world}, no collective",
                       "pool_layout": "resident pool segmented by (mode, rating group) into 2048-player chunks at ingest "
                                      "(the reference queues per group: search/worker.ex:46-66); the tick sorts by rating "
                                      "inside every group",
                       "l2": "flushed between steps (256 MiB write); pool 180 MB > L2",
                       "timed_region": "mm_tick_device: the whole tick (k_tick: hist | column scan | placement | "
                                       "epilogue in one cooperative launch), CUDA events on the engine stream; "
                                       "snapshot restore + L2 flush between steps untimed"},
            "phase_us": dict(zip(("hist", "scan", "place", "epilogue"),
                                 [round(sum(x) / len(x), 2) for x in zip(*phases)])),
            "players_per_s": total_players * args.steps / tick_s,
            "wall_ms_per_step_incl_restore": 1e3 * wall_s / args.steps,
            "roofline": {"bound": "hbm", "kernel": "k_tick" if fused else "k_hist + k_colscan + k_place + k_epilogue",
                         "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                         "bytes_per_player": B_ALG_TICK, "players_per_launch": n, "us_per_launch": 1e6 * tick_avg_s,
                         "frac_of_8000": ach / 8000.0,
                         "consumed": {"bytes_per_player": B_CONSUMED_TICK, "achieved": B_CONSUMED_TICK * n / tick_avg_s / 1e9,
                                      "frac": B_CONSUMED_TICK * n / tick_avg_s / 1e9 / peak,
                                      "note": "the tick reads the 2-byte sort key derived at ingest, not rating + mode + "
                                              "team_size (6 B): on the bytes it really consumes the fraction is lower"}},
            "cpu_baseline": cpu, "e2e": e2e, "strong": strong, "stream": stream,
            "gpu_launches": launches_per_tick * args.steps, "clocks": clocks,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, st, *last_results)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
