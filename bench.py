#!/usr/bin/env python
"""bench.py — headline benchmark of the ccx engine (BASELINE.json metric: env steps/sec).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ccx|reference] [--dump-outputs DIR]

A "step" is one pass of the fused env kernel over one batch: 65,536 games/GPU x 256 random-legal plies
(BASELINE configs[1], SURVEY.md §8d cfg 2).  See DESIGN.md §5 for every field of the JSON line.

`--dump-outputs DIR` writes what the timed path hands its caller after the last timed step (rank 0's shard), as float64
.npy files, so that two builds run with the same arguments can be compared output for output:
  state.npy       (8, G, 2)  the env state tensor (include/ccx.h layout), each uint64 word split into its low and high
                             32-bit halves (exact in float64)
  wins.npy        (2,)       the env's cumulative P1 / P2 win counters
  game_index.npy  (G,)       which games state.npy holds: all of them, or a fixed seeded sample when the whole state
                             would exceed DUMP_BYTES
The inputs depend only on the arguments (fixed seed, global game ids), so they are identical from run to run.

`--impl reference` times the UNMODIFIED Python reference (its own Board.get_valid_moves / Board.place loop, staged
as oracle/_ref/reference.zip by oracle/refrun.py) on every host core of the box; when no staged copy exists it falls
back to the C port of the same loop (oracle/ccx_oracle.c) and says so in `cpu_baseline.kind`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GAMES_PER_GPU = 65536
PLIES_PER_STEP = 256
BYTES_PER_ENV_STEP = 80          # 40 B state read + 40 B written per game-ply (SURVEY.md §8d)
SEED = 0x5EED2026
METRIC = "env_steps_per_sec"
UNIT = "env steps/s"
N_SMS, SCHEDULERS_PER_SM = 148, 4
DUMP_BYTES = 64 << 20            # --dump-outputs: upper bound on the bytes written
STEP_KERNEL = "k_step_random_wq<false, 448, 1, true>"     # the default variant of ccx_step_random (csrc/ccx_env.cu)


def workload_config(n):
    """The one `config` dict both arms print (the driver compares them)."""
    return {"workload": "cfg2 random-legal env stepping (movegen+pick+apply+win)", "games_per_gpu": n,
            "plies_per_step": PLIES_PER_STEP, "start": "Board() start position, won games restart",
            "l2": "flushed between timed steps (256 MiB write, untimed)", "parallelism": "games sharded, no collective"}


def dump_outputs(directory, state, wins):
    """state: (8, n) uint64 env state, wins: (2,) win counters -> DIR/{state,wins,game_index}.npy (see the module docstring)"""
    import numpy as np
    n = state.shape[1]
    per_game = state.shape[0] * 2 * 8 + 8                        # two float64 halves per word, plus the game's index
    keep = (DUMP_BYTES - 3 * 128 - 2 * 8) // per_game           # less three .npy headers and the win counters
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(SEED).choice(n, keep, replace=False))
    words = np.ascontiguousarray(state[:, idx]).view(np.uint32).reshape(state.shape[0], len(idx), 2)   # little-endian: lo, hi
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "state.npy"), words.astype(np.float64))
    np.save(os.path.join(directory, "wins.npy"), np.asarray(wins, dtype=np.float64))
    np.save(os.path.join(directory, "game_index.npy"), idx.astype(np.float64))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return dict(hbm_gbs=float(d["hbm_gbs"]), bf16_tflops=float(d["bf16_tflops"]), sm_max_mhz=float(d.get("sm_max_mhz", 1965.0)),
                    source="measured")
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, sm_max_mhz=1965.0, source="fallback")


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region.  NVML (nvidia_ml_py) is polled every ~2 ms so that even a
    70 ms timed region gets tens of samples; nvidia-smi (B200_PROFILING.md recipe) is the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mx, self.reasons, self.stop_flag, self.source = index, [], 0.0, set(), False, "nvml"
        self.active = threading.Event()          # samples are kept only while this is set (the timed region)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and all(x.strip().isdigit() for x in visible.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.source = "nvidia-smi"

    def _nvml_sample(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _smi_sample(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                             stdout=subprocess.PIPE, text=True, timeout=5).stdout
        s = [x.strip() for x in out.strip().split(",")]
        self.sm.append(float(s[0])); self.mx = max(self.mx, float(s[1]))
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self.stop_flag:
            if self.active.is_set():
                try:
                    self._nvml_sample() if self.nvml else self._smi_sample()
                except Exception:
                    pass
                time.sleep(0.002)
            else:
                time.sleep(0.0005)

    def summary(self):
        self.stop_flag = True
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx or None, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": self.source}


# ---- CPU legs (the only places that may execute oracle/) ---------------------------------------------------------------

def port_rate(nthreads, games, plies=PLIES_PER_STEP, step0=0):
    import oracle as orc
    st = orc.start_states(games)
    t = time.perf_counter(); orc.step_random(st, SEED, step0, plies, nthreads=nthreads); dt = time.perf_counter() - t
    return games * plies / dt


def cpu_baseline(seconds_target=10.0):
    """rank 0, N = 1: ONE host core on a bounded sample of the workload.  The unmodified Python reference when its staged copy
    is present (kind "reference"), else the C port (kind "port"); the port's one-core rate is reported beside it either way."""
    import refrun
    port = port_rate(1, 2048, 64)
    port = port_rate(1, int(min(GAMES_PER_GPU, max(2048, port * 3.0 / PLIES_PER_STEP))))
    out = {"unit": UNIT, "cores": 1, "cpu_model": refrun.cpu_model(), "host_cores": os.cpu_count(),
           "port_value": port, "port_note": "C restatement of board.py (oracle/ccx_oracle.c), 1 thread"}
    if refrun.available():
        refrun._random_steps_worker((1, 32, 0))                       # import + warm-up
        s, _, dt = refrun._random_steps_worker((2, PLIES_PER_STEP, 1))
        games = max(2, int(s / dt * seconds_target / PLIES_PER_STEP))
        s, _, dt = refrun._random_steps_worker((games, PLIES_PER_STEP, 2))
        out.update(value=s / dt, kind="reference",
                   sample="%d games x %d plies of the unmodified reference's Board loop (get_valid_moves + selfplay.py:93-98 choice + place), "
                          "1 process, %.1f s" % (games, PLIES_PER_STEP, dt))
    else:
        out.update(value=port, kind="port", sample="oracle port, 1 thread (no staged reference at oracle/_ref/reference.zip)")
    return out


def reference_extra(pool, budget_s=20.0):
    """BASELINE.md §3 items 1-4 with the unmodified reference on this box: cfg 1 greedy games (script as shipped + a 1,000-game
    Game.start loop), cfg 4 stub MCTS; single-process and all-cores figures."""
    import refrun
    out = {"cpu_model": refrun.cpu_model(), "host_cores": os.cpu_count(), "pool_processes": pool.procs}
    dt, tail = refrun.greedy_vs_greedy_script()
    out["greedy_vs_greedy_py"] = {"games": 50, "seconds": dt, "games_per_sec": 50 / dt, "processes": 1, "output_tail": tail}
    g1 = refrun._greedy_games_worker((100, 7))
    out["game_start_loop_1core"] = {"games": g1[0], "games_per_sec": g1[0] / g1[5], "plies_per_sec": g1[1] / g1[5],
                                    "plies_per_game": g1[1] / g1[0], "p1_wins": g1[2], "p2_wins": g1[3], "no_result": g1[4]}
    pool.greedy_games(pool.procs, 1)                                  # every worker imports the reference once
    g = pool.greedy_games(1000, 3)
    out["game_start_loop_all_cores"] = {"games": g["games"], "games_per_sec": g["games"] / g["seconds"], "plies_per_sec": g["plies"] / g["seconds"],
                                        "plies_per_game": g["plies"] / g["games"], "p1_wins": g["p1_wins"], "p2_wins": g["p2_wins"],
                                        "no_result": g["no_result"], "processes": pool.procs}
    s1, d1 = refrun._mcts_stub_worker((2, 175))
    sa, da = pool.mcts_stub(2 * pool.procs, 175)
    out["mcts_stub"] = {"sims_per_sec_1core": s1 / d1, "sims_per_sec_all_cores": sa / da, "sims_per_move": 175, "processes": pool.procs}
    return out


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the cfg 2 loop on the box's host cores, all of them
    (multiprocessing.Pool(os.cpu_count()), the reference's own way of going parallel: train.py:71-86).  Each step is a bounded
    sample of the 65,536-game workload sized so that warm-up + timed steps end within a few minutes."""
    if rank != 0:
        return
    import refrun
    cores = os.cpu_count() or 1
    extra = {}
    if refrun.available():
        kind = "reference"
        pool = refrun.Pool(cores)
        pool.random_steps(cores, 8, 0)                                # workers import the reference, first call
        s, _, dt = pool.random_steps(2 * cores, 64, 1)
        rate = s / dt
        budget = min(5.0, 100.0 / max(1, args.steps + args.warmup))   # seconds per step
        games = int(max(cores, min(GAMES_PER_GPU, rate * budget / PLIES_PER_STEP)))
        games -= games % cores
        for w in range(args.warmup):
            pool.random_steps(games, PLIES_PER_STEP, 100 + w)
        total = wins = 0
        t = time.perf_counter()
        for k in range(args.steps):
            s, w, _ = pool.random_steps(games, PLIES_PER_STEP, 1000 + k)
            total += s; wins += w
        dt = time.perf_counter() - t
        value = total / dt
        sample = ("%d games x %d plies per step of the unmodified reference's Board loop (get_valid_moves + selfplay.py:93-98 choice + "
                  "Board.place), multiprocessing.Pool(%d); bounded sample of the %d-game workload" % (games, PLIES_PER_STEP, cores, GAMES_PER_GPU))
        if not args.no_extra:
            try:
                extra["reference_cpu"] = reference_extra(pool)
            except Exception as e:                                    # never lose the headline line to a side measurement
                extra["reference_cpu_error"] = repr(e)
        pool.close()
        extra["port_all_threads"] = {"value": port_rate(cores, 8192), "unit": UNIT, "threads": cores,
                                     "note": "C restatement of the same loop (oracle/ccx_oracle.c), for scale"}
    else:
        kind = "port"
        import oracle as orc
        games = GAMES_PER_GPU                                         # the whole workload: ~2 s per step on 16 threads
        st = orc.start_states(games)
        for w in range(args.warmup):
            st, _, _ = orc.step_random(st, SEED, w * PLIES_PER_STEP, PLIES_PER_STEP, nthreads=cores)
        t = time.perf_counter()
        for k in range(args.steps):
            st, _, _ = orc.step_random(st, SEED, (args.warmup + k) * PLIES_PER_STEP, PLIES_PER_STEP, nthreads=cores)
        dt = time.perf_counter() - t
        value = games * PLIES_PER_STEP * args.steps / dt
        sample = ("%d games x %d plies per step, oracle port (C restatement of board.py) on %d threads; no staged reference under "
                  "oracle/_ref/reference.zip" % (games, PLIES_PER_STEP, cores))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(GAMES_PER_GPU),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "per_core": value / cores,
                         "cpu_model": refrun.cpu_model()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}
    if extra:
        line["extra"] = extra
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ccx", choices=["ccx", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--games", type=int, default=GAMES_PER_GPU, help="games per GPU (BASELINE config: 65536)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as .npy files into DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ccx":
        ap.error("--dump-outputs applies to the GPU path (--impl ccx)")
    args.warmup = max(args.warmup, 3) if args.impl == "ccx" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from chinesecheckersagent_b200.engine import BatchedEnv, Engine, HostEnv

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    eng = Engine(local_rank)
    n = args.games
    env = BatchedEnv(n, engine=eng, seed=SEED, game_id0=rank * n)     # global game ids: sharding-invariant RNG
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        env.step_random(PLIES_PER_STEP)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.active.set()
    for a, b in evs:
        flush.fill_(1)                      # L2 flush between timed iterations (not timed)
        a.record()
        env.step_random(PLIES_PER_STEP)     # torch's current stream == the handle's stream
        b.record()
    barrier()
    sampler.active.clear()
    launches = eng.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env.numpy_state(), env.wins.cpu().numpy())
    per_step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = torch.tensor([sum(per_step_ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms.item()) / 1e3
    steps_total = world * n * PLIES_PER_STEP * args.steps
    value = steps_total / total_s

    # ---- end-to-end through the host-buffer C-ABI (pinned host state in, state + win counters out)
    host = HostEnv(engine=eng)
    st_pinned = torch.from_numpy(np.ascontiguousarray(env.numpy_state()).view(np.int64)).pin_memory()
    st_np = st_pinned.numpy().view(np.uint64)
    wins = np.zeros(2, dtype=np.uint64)
    e2e_steps = max(3, min(args.steps, 10))
    host.step_random(st_np, PLIES_PER_STEP, seed=SEED, step0=0, game_id0=rank * n, wins=wins)
    barrier()
    sampler.active.set()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        host.step_random(st_np, PLIES_PER_STEP, seed=SEED, step0=(k + 1) * PLIES_PER_STEP, game_id0=rank * n, wins=wins)
    torch.cuda.synchronize()
    e2e_t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    sampler.active.clear()
    clocks = sampler.summary() if rank == 0 else None
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * PLIES_PER_STEP * e2e_steps / float(e2e_t.item())
    h2d = n * 40 + 16
    d2h = n * 40 + 16

    peaks = measured_peaks()
    extra = {}
    if not args.no_extra:
        # saturated rate of the step kernel: the same 256-ply launch on larger batches (65,536 games fill 13.8 warps per SM)
        sweep = {}
        for m in (GAMES_PER_GPU, 2 * GAMES_PER_GPU, 4 * GAMES_PER_GPU, 8 * GAMES_PER_GPU, 16 * GAMES_PER_GPU):
            e2 = BatchedEnv(m, engine=eng, seed=SEED, game_id0=rank * m)
            e2.step_random(PLIES_PER_STEP)
            barrier()
            ts = []
            for _ in range(3):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                flush.fill_(1); a.record(); e2.step_random(PLIES_PER_STEP); b.record()
                ts.append((a, b))
            torch.cuda.synchronize()
            ms = sum(a.elapsed_time(b) for a, b in ts) / 3
            sweep[str(m)] = {"env_steps_per_sec_per_gpu": m * PLIES_PER_STEP / (ms * 1e-3), "ms_per_launch": ms}
            del e2
        extra["games_per_gpu_sweep"] = sweep
        try:
            from chinesecheckersagent_b200 import bench_extra
            extra.update(bench_extra.run(eng, rank, world, barrier, peak_gbs=peaks["hbm_gbs"], peak_tflops=peaks["bf16_tflops"]))
        except ImportError:
            pass

    if rank == 0:
        launch_ms = sum(per_step_ms) / len(per_step_ms)
        achieved = BYTES_PER_ENV_STEP * n * PLIES_PER_STEP / (launch_ms * 1e-3) / 1e9
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                prof = json.load(f)
        except Exception:
            pass
        traffic = prof.get("k_step_random_flat")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": workload_config(n),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                         "traffic": traffic, "peak_source": peaks["source"], "kernel": STEP_KERNEL,
                         "algorithmic_bytes_per_launch": BYTES_PER_ENV_STEP * n * PLIES_PER_STEP, "launch_ms": launch_ms,
                         "traffic_source": prof.get("source")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "ccx_step_random_host (pinned host state in/out)", "steps": e2e_steps},
            "gpu_launches": launches, "clocks": clocks,
        }
        # the roofline that actually binds this kernel (state stays in registers for all 256 plies, DRAM traffic is ~500x below the
        # algorithmic bytes): warp instructions issued per second against 148 SMs x 4 schedulers x 1 instruction per clock
        winst = prof.get("k_step_random_flat_warp_insts")
        if winst and n == GAMES_PER_GPU:
            f_mhz = (clocks or {}).get("sm_mhz") or peaks["sm_max_mhz"]
            ach_i = winst / (launch_ms * 1e-3)
            peak_i = N_SMS * SCHEDULERS_PER_SM * f_mhz * 1e6
            line["roofline_issue"] = {"bound": "issue", "achieved": ach_i, "peak": peak_i, "unit": "warp-instr/s", "frac": ach_i / peak_i,
                                      "warp_insts_per_launch": winst, "sm_mhz": f_mhz, "kernel": STEP_KERNEL,
                                      "source": "smsp__inst_executed.sum of the ncu capture named in roofline.traffic_source; launch time measured live"}
        # the unit this kernel keeps busiest: the shared-memory data pipe (the lanes' random reads of the jump tables; half of the
        # wavefronts are bank conflicts) — wavefronts per second against one wavefront per SM and clock
        wav = prof.get("k_step_random_flat_smem_wavefronts")
        if wav and n == GAMES_PER_GPU:
            f_mhz = (clocks or {}).get("sm_mhz") or peaks["sm_max_mhz"]
            ach_w = wav / (launch_ms * 1e-3)
            peak_w = N_SMS * f_mhz * 1e6
            line["roofline_smem"] = {"bound": "shared-memory data pipe", "achieved": ach_w, "peak": peak_w, "unit": "wavefronts/s", "frac": ach_w / peak_w,
                                     "wavefronts_per_launch": wav, "bank_conflict_wavefronts_per_launch": prof.get("k_step_random_flat_smem_conflicts"),
                                     "sm_mhz": f_mhz, "kernel": STEP_KERNEL,
                                     "source": "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum of the ncu capture named in roofline.traffic_source; launch time measured live"}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
            if not args.no_extra:
                # the reference's other CPU figures (cfg 1 / cfg 4) on this box's host cores, same run (BASELINE.md §3)
                try:
                    import refrun
                    if refrun.available():
                        pool = refrun.Pool(os.cpu_count(), spawn=True)        # CUDA is initialised in this process: spawn, not fork
                        extra["reference_cpu"] = reference_extra(pool)
                        s, _, dt = pool.random_steps(4 * pool.procs, PLIES_PER_STEP, 5)
                        extra["reference_cpu"]["random_env_steps_per_sec_all_cores"] = s / dt
                        pool.close()
                except Exception as e:
                    extra["reference_cpu_error"] = repr(e)
        if extra:
            line["extra"] = extra
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
