#!/usr/bin/env python
"""bench.py — throughput of the batched hot paths on N B200s (one process per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ekf|pf|mpc]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch of synthetic input (BASELINE.json configs):
  ekf (headline, configs[1]): 2^20 agents x 1 EKF update per GPU          metric: EKF updates/s
  pf  (configs[2]):           2^20 particles x 8 landmarks per GPU        metric: particle updates/s
  mpc (configs[3]/[4]):       65 536 agents, T=20 per GPU                 metric: MPC solves/s
The default run prints ONE JSON line whose headline is the EKF config.  BASELINE.json's metric is "EKF updates/sec
& MPC solves/sec", so the MPC (and PF) figures of the same run are FIRST-CLASS in that line: `roofline.mpc`,
`e2e.mpc`, `cpu_baseline.mpc` (same for `pf`), `config.mpc_solves_per_s`, and with --gpus N > 1 BASELINE
configs[4] as written (`config5`: 2^20 MPC agents sharded over the N GPUs, one stats all-gather per call).  The
full per-workload records stay under "extra".
Weak scaling (headline): per-GPU work is fixed, shard r holds global indices [r*n, (r+1)*n) of the
index-addressed generators; the only inter-GPU traffic is one all-gather of 8 doubles per rank, issued by
libcrb's own NCCL communicator (crb_gather_stats) INSIDE the captured graph.

Timing rules followed: W >= 3 warm-up steps; inputs rotate over 3 buffer sets whose total exceeds the
126 MB L2; the K steps (+ stats tail + all-gather) are captured once in a CUDA graph, replayed once untimed, then
once as the timed window: exactly K timed steps between two CUDA events on the launching stream, bracketed by
barrier + synchronize, the window's time maxed over ranks; `ms_per_step` is the window / K; SM clocks sampled with
nvidia-smi during the timed region.

--dump-outputs DIR writes, after the timed steps, what the headline's last timed step returned to its caller
(rank 0's shard): DIR/ekf_x.npy, the filtered states of all 2^20 agents, and DIR/ekf_P.npy, the covariances of a
fixed seeded sample of 2^17 agents (DIR/ekf_P_agents.npy holds their indices), float32 (the indices float64),
25 MB in all.  Inputs are seeded, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the CPU restatement of the reference (oracle/, the only implementation of the
path that can run here: Eigen/IPOPT are absent) on the box's host cores with all threads.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: nothing is compiled or cached in it at run time

EKF_N = 1 << 20
PF_N = int(os.environ.get("CRB_BENCH_PF_N", 1 << 20))     # diagnostics only: the contract workload is 2^20 x 8
PF_LM = int(os.environ.get("CRB_BENCH_PF_LM", 8))
MPC_N = int(os.environ.get("CRB_BENCH_MPC_N", 1 << 16))    # diagnostics only: the contract workload is 2^16
MPC_T = 20
MPC_ITER, MPC_DUTH, MPC_LS = 50, 1e-4, 4   # IPOPT's max_iter (:326); tight du so the NLP converges
EKF_BYTES = 176       # read x4 P16 z2 u2, write x4 P16 (f32)            SURVEY §8 d-3
PF_BYTES = 48         # read px4 w1 noise2, write px4 w1                  SURVEY §8 d-4
MPC_BYTES = 344 + 472 # read x0 4 + xref 80, write sol 118 + u0 2 (+cost,status,iters 3) f32 ~ 828
NSETS = 3


PINNED_CPUS = [0]


def host_threads() -> int:
    """All host cores this process may use.  torchrun exports OMP_NUM_THREADS=1, which would silently make the
    CPU arm single-threaded; the oracle takes an explicit thread count instead.  Once the CPU arm has pinned the
    process (cpu_pin_one_numa_node) the count is the size of THAT set: with OMP_PROC_BIND the OpenMP runtime binds
    the calling thread to a single core, so the affinity mask read later would say 1."""
    if PINNED_CPUS[0]:
        return PINNED_CPUS[0]
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)", d
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)", {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[4 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_setup(n_gpus: int):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"     # keep stdout to the one JSON line
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    if world != n_gpus:
        raise SystemExit(f"--gpus {n_gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    return rank, world, local


def barrier_sync(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms: float, world: int) -> float:
    import torch
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def max_over_ranks_cpu(ms: float, world: int) -> float:
    """gloo flavour of max_over_ranks for the CPU multi-process tests."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_stats(stats, world, eng=None, out=None):
    """The single collective of the data path: all-gather of CRB_STATS_LEN doubles per rank.  On the GPU it is
    libcrb's own NCCL communicator (crb_gather_stats, capturable in a CUDA graph); the torch.distributed form
    is what the CPU (gloo) tests of the host logic use."""
    import torch
    if eng is not None and (world == 1 or eng.world == world):
        return eng.gather_stats(stats, out=out)
    if world == 1:
        return stats.unsqueeze(0)
    import torch.distributed as dist
    out = torch.empty(world * stats.numel(), dtype=stats.dtype, device=stats.device)
    dist.all_gather_into_tensor(out, stats.contiguous().view(-1))
    return out.view(world, stats.numel())


def comm_setup(eng, rank, world):
    """Bootstrap libcrb's communicator: rank 0 creates the NCCL unique id, torch.distributed (already up for the
    barrier / max-over-ranks plumbing) carries the 128 bytes."""
    if world == 1:
        return
    import torch
    import torch.distributed as dist
    from cpprobotics_b200 import _lib as L
    buf = torch.zeros(L.CRB_COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
    if rank == 0:
        buf.copy_(torch.frombuffer(bytearray(eng.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(buf, 0)
    eng.comm_init(world, rank, bytes(buf.cpu().numpy().tobytes()))


NUMA_INFO = {}


def gpu_numa_cpus(device_index=0):
    """CPUs of the NUMA node the GPU hangs off (PCI bus id from nvidia-smi -> sysfs numa_node -> cpulist), or None.
    The result (or the reason it is unknown) is kept in NUMA_INFO and reported in the JSON line."""
    if device_index in NUMA_INFO:
        return NUMA_INFO[device_index].get("cpus")
    info = {"node": None, "cpus": None, "why": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        rows = [l.split(",") for l in out.strip().splitlines() if "," in l]
        phys = device_index
        if visible:
            ids = [v.strip() for v in visible.split(",")]
            if device_index < len(ids) and ids[device_index].isdigit():
                phys = int(ids[device_index])
        bus = next((r[1].strip() for r in rows if int(r[0]) == phys), None)
        if bus is None:
            raise RuntimeError("GPU not listed by nvidia-smi")
        dom, rest = bus.split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            raise RuntimeError("numa_node = -1 (single node or not exposed)")
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        info.update(node=node, cpus=cpus)
    except Exception as exc:
        info["why"] = str(exc)[:120]
    NUMA_INFO[device_index] = info
    return info["cpus"]


def numa_pinned(a, device_index=0):
    """Pinned host copy of `a` allocated (and first touched) while this thread runs on the CPUs of the GPU's NUMA
    node (eight GPUs pulling from one node's DRAM was r1's e2e limiter at N = 8)."""
    import torch
    old = None
    cpus = gpu_numa_cpus(device_index)
    try:
        if cpus:
            old = os.sched_getaffinity(0)
            use = cpus & old
            if use:
                os.sched_setaffinity(0, use)
            else:
                old = None
    except Exception:
        old = None
    try:
        t = torch.empty(a.shape, dtype=torch.from_numpy(a).dtype).pin_memory()
        t.copy_(torch.from_numpy(a))
    finally:
        if old is not None:
            os.sched_setaffinity(0, old)
    return t


def pinned(a):
    import torch
    return numa_pinned(np.ascontiguousarray(a), torch.cuda.current_device())


# =========================================================================================================
# workloads: each returns a dict with value / ms_per_step / roofline / e2e / cpu_baseline pieces
# =========================================================================================================
LAST_TIMING = {}


def time_device_steps(step_fn, steps, warmup, world, after_fn=None, eng=None, graph=True):
    """W untimed steps, then the K steps (+ the optional tail: stats reduction and the all-gather) captured ONCE
    into a CUDA graph.  After barrier + synchronize the graph is replayed once untimed (upload and first-launch
    costs) and, enqueued right behind it, once more as the timed window: exactly K timed steps between a pair of
    CUDA events on the launching stream, then barrier + synchronize, the window's time maxed over ranks.  Returns
    (window ms, mode); LAST_TIMING holds the record.  If capture is not possible the K steps are enqueued directly,
    once, timed."""
    import torch
    for k in range(warmup):
        step_fn(k)
    if after_fn is not None:
        after_fn()
    mode = "stream"
    g = None
    if graph and eng is not None:
        try:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                eng.bind_current_stream()
                for k in range(steps):
                    step_fn(warmup + k)
                if after_fn is not None:
                    after_fn()
            eng.bind_current_stream()
            mode = "cuda_graph"
        except Exception as exc:            # pragma: no cover - depends on driver / torch
            sys.stderr.write(f"graph capture failed ({exc}); timing direct launches\n")
            eng.bind_current_stream()
            g = None
    barrier_sync(world)
    if g is not None:
        g.replay()      # untimed; the GPU is still running it when e0 is reached, so no launch latency is timed
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if g is not None:
        g.replay()
    else:
        for k in range(steps):
            step_fn(warmup + k)
        if after_fn is not None:
            after_fn()
    e1.record()
    barrier_sync(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    LAST_TIMING.clear()
    LAST_TIMING.update(timed_steps=int(steps), ms=ms, mode=mode)
    return ms, mode


def timing_record(steps):
    t = dict(LAST_TIMING)
    return dict(timed_steps=t.get("timed_steps"), ms_per_step=t.get("ms", 0.0) / steps, launch=t.get("mode"))


def time_host_steps(step_fn, steps, warmup, world):
    import torch
    for k in range(max(1, min(warmup, 2))):
        step_fn(k)
    barrier_sync(world)
    t0 = time.perf_counter()
    for k in range(steps):
        step_fn(k)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    barrier_sync(world)
    return max_over_ranks(ms, world)


def cpu_pin_one_numa_node():
    """CPU arm hygiene (r1's CPU figures swung 6x between boxes): restrict this process to the CPUs of ONE NUMA
    node (the one with the most CPUs in our affinity mask) before the OpenMP runtime starts, and ask it to bind
    threads to cores.  Returns (restore_fn, description)."""
    old = os.sched_getaffinity(0)
    best, best_node = set(), None
    try:
        for d in sorted(os.listdir("/sys/devices/system/node")):
            if not d.startswith("node") or not d[4:].isdigit():
                continue
            cpus = set()
            for part in open(f"/sys/devices/system/node/{d}/cpulist").read().strip().split(","):
                if not part:
                    continue
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            use = cpus & old
            if len(use) > len(best):
                best, best_node = use, d
    except OSError:
        pass
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")

    def restore():
        PINNED_CPUS[0] = 0
        os.sched_setaffinity(0, old)
    if best and len(best) < len(old):
        os.sched_setaffinity(0, best)
        PINNED_CPUS[0] = len(best)
        return restore, f"{len(best)} CPUs of NUMA {best_node} (of {len(old)} allowed)"
    PINNED_CPUS[0] = len(old)
    return restore, f"{len(old)} allowed CPUs (single NUMA node or no topology information)"


def cpu_time(fn, units_per_call, budget_s=6.0, min_passes=5):
    """Bounded CPU sample: >= 5 timed passes (more until ~budget_s), each timed on its own; returns the MEDIAN
    rate in units/s plus the spread, so that one descheduled pass does not move the figure."""
    fn()  # warm caches / thread pool
    ts = []
    t_all = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
        el = time.perf_counter() - t_all
        if len(ts) >= min_passes and el >= budget_s:
            break
        if el > 4 * budget_s and len(ts) >= 2:
            break
    ts = np.array(ts)
    spread = dict(passes=int(ts.size), fastest=units_per_call / ts.min(), slowest=units_per_call / ts.max())
    CPU_SPREAD.append(spread)
    return units_per_call / float(np.median(ts)), int(ts.size), float(ts.sum())


CPU_SPREAD = []


def tuned_threads(fn_thr, label=""):
    """Thread count for a CPU arm.  "All the cores in the affinity mask" is not always the fastest choice on
    shared hosts (r1: 128 OpenMP threads measured 10x SLOWER than 64), so the arm times cores, 3/4, 1/2 and 1/4
    of the mask, FIVE passes each, and keeps the team with the best median -- the baseline is the best the host
    can do, not a strawman, and not a two-sample accident."""
    cores = host_threads()
    cand = sorted({max(1, cores), max(1, 3 * cores // 4), max(1, cores // 2), max(1, cores // 4)},
                  reverse=True)
    best, best_t = cand[0], None
    for c in cand:
        fn_thr(c)                       # warm this team size
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            fn_thr(c)
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        if best_t is None or t < best_t:
            best, best_t = c, t
    return best, cores


def best_effort(fn, units, budget_s=2.0):
    """BASELINE.md B2: the same CPU code built -O3 -march=x86-64-v3 -ffp-contract=fast (oracle/lib/
    liboracle_fast.so), same thread count; a timing arm only.  None when that build or AVX2/FMA is missing."""
    from oracle import oracle as O
    if not O.use_library("fast"):
        O.use_library("faithful")
        return None
    try:
        v, _, _ = cpu_time(fn, units, budget_s=budget_s, min_passes=3)
    finally:
        O.use_library("faithful")
    return v


def as_shipped_O0(fn, units, budget_s=1.0):
    """BASELINE.md B0: the reference builds without optimisation (CMakeLists.txt:5): the same restatement at -O0,
    recorded once for context."""
    from oracle import oracle as O
    if not O.use_library("O0"):
        O.use_library("faithful")
        return None
    try:
        v, _, _ = cpu_time(fn, units, budget_s=budget_s, min_passes=2)
    finally:
        O.use_library("faithful")
    return v


def dump_ekf(out_dir, x, P):
    """The state of every agent and the covariance of a fixed seeded sample of 2^17 agents (P of all 2^20 would be
    64 MB on its own)."""
    import torch
    agents = np.sort(np.random.default_rng(20).choice(x.shape[1], 1 << 17, replace=False))
    idx = torch.from_numpy(agents).to(P.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("ekf_x", x.cpu().numpy()), ("ekf_P", P.index_select(1, idx).cpu().numpy()),
                    ("ekf_P_agents", agents.astype(np.float64))):
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def bench_ekf(eng, rank, world, steps, warmup, with_cpu, dump_dir=None):
    import torch
    from cpprobotics_b200 import synth
    n = EKF_N
    dev = torch.device("cuda", torch.cuda.current_device())
    host = synth.ekf_inputs(n, i0=rank * n)
    sets = []
    for s in range(NSETS):   # identical contents, distinct memory: only residency matters
        sets.append(tuple(torch.from_numpy(a).to(dev) for a in host))
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    table = torch.zeros((world, 8), dtype=torch.float64, device=dev)

    def step(k):
        x, P, z, u = sets[k % NSETS]
        eng.ekf_estimation(x, P, z, u)

    def after():
        eng.stats_reduce(sets[0][0][0], i0=rank * n, out=stats)   # summary of the x field
        gather_stats(stats, world, eng, out=table)                # libcrb's NCCL all-gather, inside the graph

    ms, mode = time_device_steps(step, steps, warmup, world, after, eng=eng)
    timing = timing_record(steps)
    if dump_dir is not None and rank == 0:
        dump_ekf(dump_dir, *sets[(warmup + steps - 1) % NSETS][:2])    # step() updates x, P in place
    launches = steps + 2 + (1 if world > 1 else 0)   # K filter kernels + two stats-reduction kernels (+ NCCL's)
    value = world * n * steps / (ms * 1e-3)
    # roofline of the dominant kernel (one launch per step): algorithmic bytes / avg launch duration,
    # measured separately WITHOUT the stats tail so that it is the kernel alone.
    ms_k, _ = time_device_steps(step, steps, 3, world, eng=eng)
    k_timing = timing_record(steps)
    peak, peak_src, _ = peaks()
    achieved = EKF_BYTES * n * steps / (ms_k * 1e-3) / 1e9
    copy_gbs = copy_ceiling_gbs()
    # e2e (a): one-shot through the host-pointer C-ABI entry: pinned host buffers, all 176 B per update cross
    # PCIe every step
    hx, hP, hz, hu = (pinned(a) for a in host)
    e_steps = max(3, min(steps, 10))
    ms_e = time_host_steps(lambda k: eng.ekf_estimation_host(hx, hP, hz, hu), e_steps, warmup, world)
    # e2e (b): the reference's own loop shape (:171-183): x, P stay on the device, each step ships z, u (16 B)
    # in and x (16 B) out, pipelined over two sets of pinned buffers
    trk = eng.ekf_track_open(host[0], host[1])
    zs = [pinned(host[2]) for _ in range(2)]
    us = [pinned(host[3]) for _ in range(2)]
    xo = [pinned(np.zeros((4, n), np.float32)) for _ in range(2)]
    s_steps = max(10, steps)

    def track(k):
        eng.ekf_track_step(trk, zs[k & 1], us[k & 1], x_out=xo[k & 1], async_=True)
    for k in range(4):
        track(k)
    eng.ekf_track_sync(trk)
    barrier_sync(world)
    t0 = time.perf_counter()
    for k in range(s_steps):
        track(k)
    eng.ekf_track_sync(trk)
    ms_s = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
    barrier_sync(world)
    eng.ekf_track_close(trk)
    out = dict(value=value, ms=ms / steps, launches=launches, launch_mode=mode, timing=timing,
               roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s",
                             frac=achieved / peak, traffic=traffic_for("ekf"), peak_source=peak_src,
                             kernel="crb_ekf_step_kernel",
                             algorithmic_bytes_per_launch=EKF_BYTES * n,
                             ms_per_launch=k_timing["ms_per_step"],
                             copy_gbs_same_run=copy_gbs, frac_of_copy_same_run=achieved / copy_gbs),
               e2e=dict(value=world * n * e_steps / (ms_e * 1e-3), unit="updates/s",
                        h2d_bytes_per_step=96 * n, d2h_bytes_per_step=80 * n,
                        path="crb_ekf_step_batched_host on pinned buffers (NUMA-local to the GPU): kernel reads/"
                             "writes host memory over PCIe directly (zero-copy), synchronous per step",
                        resident_state=dict(
                            value=world * n * s_steps / (ms_s * 1e-3), unit="updates/s",
                            h2d_bytes_per_step=16 * n, d2h_bytes_per_step=16 * n, steps=s_steps,
                            path="crb_ekf_track_step: x, P resident in HBM across steps (the reference's loop, "
                                 ":171-183), z,u read over PCIe by the kernel, x returned through a snapshot copy "
                                 "overlapped with the next step")))
    if with_cpu and rank == 0:
        out["cpu_baseline"] = cpu_ekf(host)
    return out


def cpu_ekf(host=None):
    from cpprobotics_b200 import synth
    from oracle import oracle as O
    n = EKF_N
    x, P, z, u = host if host is not None else synth.ekf_inputs(n)
    x, P = x.copy(), P.copy()
    CPU_SPREAD.clear()
    thr, mask = tuned_threads(lambda c: O.ekf_step_batched(x, P, z, u, nthreads=c, inplace=True))
    v, calls, el = cpu_time(lambda: O.ekf_step_batched(x, P, z, u, nthreads=thr, inplace=True), n,
                            budget_s=5.0)
    spread = CPU_SPREAD[-1]
    m = 1 << 18                                   # SURVEY d-7: the same code on ONE core
    x1, P1, z1, u1 = (np.ascontiguousarray(a[:, :m]) for a in (x, P, z, u))
    v1, _, _ = cpu_time(lambda: O.ekf_step_batched(x1, P1, z1, u1, nthreads=1, inplace=True), m, budget_s=1.0,
                        min_passes=3)
    vb = best_effort(lambda: O.ekf_step_batched(x, P, z, u, nthreads=thr, inplace=True), n)
    v0 = as_shipped_O0(lambda: O.ekf_step_batched(x1, P1, z1, u1, nthreads=1, inplace=True), m)
    return dict(value=v, unit="updates/s", cores=thr, kind="port", single_core_value=v1, best_effort_value=vb,
                b0_O0_single_core_value=v0, spread=spread,
                sample=f"median of {calls} passes x {n} agents x 1 step, oracle/crb_oracle.c -O2 -ffp-contract=off, "
                       f"OpenMP {thr} threads bound to cores (best median of 5 passes at 1/4..1 x the {mask}-cpu "
                       f"mask), {el:.1f} s")


def bench_pf(eng, rank, world, steps, warmup, with_cpu):
    import torch
    from cpprobotics_b200 import synth
    n = PF_N
    dev = torch.device("cuda", torch.cuda.current_device())
    host = synth.pf_inputs(n, i0=rank * n, n_total=world * n)
    lm = synth.pf_landmarks(PF_LM)
    sets = [tuple(torch.from_numpy(a).to(dev) for a in host) for _ in range(NSETS + 3)]  # 6 x 29 MB

    def step(k):
        px, pw, noise = sets[k % len(sets)]
        pw.fill_(1.0 / (world * n))     # keep weights in the normal range across repeated steps
        eng.pf_predict_weight(px, pw, noise, lm)

    def step_nofill(k):
        px, pw, noise = sets[k % len(sets)]
        eng.pf_predict_weight(px, pw, noise, lm)

    ms_k, _ = time_device_steps(step_nofill, steps, warmup, world, eng=eng)
    value = world * n * steps / (ms_k * 1e-3)
    peak, peak_src, _ = peaks()
    achieved = PF_BYTES * n * steps / (ms_k * 1e-3) / 1e9
    hpx, hpw, hno = (pinned(a) for a in host)
    e_steps = max(3, min(steps, 10))
    ms_e = time_host_steps(lambda k: eng.pf_predict_weight_host(hpx, hpw, hno, lm), e_steps, warmup,
                           world)
    out = dict(metric="PF particle updates/sec (predict+weight, 8 landmarks)", value=value,
               unit="particles/s", ms_per_step=ms_k / steps, timing=timing_record(steps),
               config=dict(workload="pf_predict_weight_2^20_particles_8_landmarks_per_gpu",
                           l2=f"{len(sets)} rotating buffer sets, {len(sets) * 29} MB > 126 MB L2"),
               roofline=dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s",
                             frac=achieved / peak, traffic=traffic_for("pf"), peak_source=peak_src,
                             kernel="crb_pf_predict_weight_lean_kernel",
                             algorithmic_bytes_per_launch=PF_BYTES * n),
               e2e=dict(value=world * n * e_steps / (ms_e * 1e-3), unit="particles/s",
                        h2d_bytes_per_step=28 * n, d2h_bytes_per_step=20 * n))
    if with_cpu and rank == 0:
        out["cpu_baseline"] = cpu_pf(host, lm)
    return out


def bench_pf_iteration(eng, rank, world, steps, warmup):
    """Row f-2: one complete filter iteration per step = crb_pf_step: predict+weight (:81-102), normalise +
    estimate + covariance (:104-107), Neff and low-variance resampling decided on the device (:120-148, forced
    every step with nth = n), particle arrays ping-ponged.  No host round trip, so the K iterations are captured
    in a CUDA graph like every other workload.  With world > 1 the filter is sharded: the weight sum and the
    moments are all-reduced inside libcrb and particles are not resampled across GPUs."""
    import torch
    from cpprobotics_b200 import synth
    n = 1 << 20
    dev = torch.device("cuda", torch.cuda.current_device())
    px, pw, noise = (torch.from_numpy(a).to(dev) for a in synth.pf_inputs(n, i0=rank * n, n_total=world * n))
    lm = synth.pf_landmarks(PF_LM)
    bufs = [px, torch.empty_like(px)]
    res = torch.zeros(24, dtype=torch.float64, device=dev)

    def step(k):
        eng.pf_step(bufs[k & 1], pw, bufs[(k + 1) & 1], noise, lm, resample_seed=k, nth=float(n), result=res)
    steps += steps & 1          # an even number of steps per replay keeps the ping-pong consistent across replays
    ms, mode = time_device_steps(step, steps, warmup + (warmup & 1), world, eng=eng)
    r = res.cpu().numpy()
    return dict(metric="PF filter iterations (predict+weight, estimate, resample) x particles per second",
                value=world * n * steps / (ms * 1e-3), unit="particles/s", ms_per_step=ms / steps,
                timing=timing_record(steps),
                config=dict(workload="pf_full_iteration_2^20_particles_per_gpu (crb_pf_step)", steps=steps,
                            resampled_last_step=bool(r[22] == 1.0), neff_last_step=float(r[21]), launch=mode,
                            note="3 kernels per iteration (predict+weight leaving the CTA weight sums; normalise + scan + "
                                 "moments of the normalised weights; gather with the block-offset scan and the resampling "
                                 "decision in its prologue and one extra CTA for xEst / PEst), programmatic dependent "
                                 "launch, no host synchronisation, no device copy; round 1 "
                                 "was 10 kernels, 2 synchronous read-backs and a 16 MB copy (135 us)"))


def cpu_pf(host=None, lm=None):
    from cpprobotics_b200 import synth
    from oracle import oracle as O
    n = PF_N
    px, pw, noise = host if host is not None else synth.pf_inputs(n)
    lm = lm if lm is not None else synth.pf_landmarks(PF_LM)
    px, pw0 = px.copy(), pw.copy()
    pw = pw0.copy()

    def one_thr(c):
        pw[:] = pw0          # keep the weights in the normal range across repeated steps
        O.pf_predict_weight_batched(px, pw, noise, lm, nthreads=c, inplace=True)
    thr, mask = tuned_threads(one_thr)
    v, calls, el = cpu_time(lambda: one_thr(thr), n, budget_s=4.0)
    vb = best_effort(lambda: one_thr(thr), n)
    return dict(value=v, unit="particles/s", cores=thr, kind="port", best_effort_value=vb,
                sample=f"{calls} x {n} particles x {PF_LM} landmarks, oracle/crb_oracle.c, OpenMP {thr} "
                       f"threads (fastest of 1/4..1 x the {mask}-cpu mask), {el:.1f} s")


def mpc_flops(iters_sum, n, T):
    """Executed-work flop model (DESIGN.md §MPC): per outer iteration one backward sweep (~470 flop /
    stage, structured) and ~1.2 forward sweeps (~150 flop / stage incl. polynomial sin/cos)."""
    return iters_sum * (T - 1) * (470.0 + 1.2 * 150.0)


FP32_PEAK = {}


def fp32_peak(eng):
    """Non-tensor fp32 FMA rate MEASURED in this run on this GPU (crb_probe_fp32_peak); nominal as fallback."""
    if "v" not in FP32_PEAK:
        sm_max = float(peaks()[2].get("sm_max_mhz", 1965.0))
        nominal = 148 * 128 * 2 * sm_max * 1e6 / 1e12
        try:
            v = eng.probe_fp32_peak()
            FP32_PEAK.update(v=v, src=f"measured in this run: crb_probe_fp32_peak (register-only FFMA kernel, best of 5); "
                                      f"nominal 148 SM x 128 lanes x 2 x {sm_max:.0f} MHz = {nominal:.1f}")
        except Exception as exc:   # pragma: no cover
            FP32_PEAK.update(v=nominal, src=f"nominal (probe failed: {exc})")
    return FP32_PEAK["v"], FP32_PEAK["src"]


def bench_mpc(eng, rank, world, steps, warmup, with_cpu, n=None, label=None, with_e2e=True):
    """One step = one crb_mpc_solve_batched over this rank's n agents + the per-shard cost statistics + ONE
    all-gather of them (BASELINE configs[3] / [4]; caller loop src/model_predictive_control.cpp:372-378)."""
    import torch
    from cpprobotics_b200 import mpc_default_params, synth
    n, T = (MPC_N if n is None else n), MPC_T
    dev = torch.device("cuda", torch.cuda.current_device())
    course = synth.mpc_course()
    st, pind = synth.mpc_states(n, i0=rank * n, course=course)
    xref, _ = synth.mpc_xref_numpy(st, pind, T, course=course)
    prm = mpc_default_params()
    prm.max_iter, prm.du_th, prm.max_ls = MPC_ITER, MPC_DUTH, MPC_LS
    nsol = 4 * T + 2 * (T - 1)
    sets = [(torch.from_numpy(st).to(dev), torch.from_numpy(xref).to(dev)) for _ in range(NSETS)]
    sol = torch.empty((nsol, n), dtype=torch.float32, device=dev)
    u0 = torch.empty((2, n), dtype=torch.float32, device=dev)
    cost = torch.empty(n, dtype=torch.float32, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    iters = torch.empty(n, dtype=torch.int32, device=dev)
    stats = torch.zeros(8, dtype=torch.float64, device=dev)
    table = torch.zeros((world, 8), dtype=torch.float64, device=dev)

    def step(k):
        s, xr = sets[k % NSETS]
        eng.mpc_solve(s, xr, T, prm, sol=sol, u0=u0, cost=cost, status=status, iters=iters)
        eng.stats_reduce(cost, status, iters, i0=rank * n, out=stats)
        gather_stats(stats, world, eng, out=table)     # config 5: the gather of cost stats, every call

    def step_kernel_only(k):
        s, xr = sets[k % NSETS]
        eng.mpc_solve(s, xr, T, prm, sol=sol, u0=u0, cost=cost, status=status, iters=iters)

    ms, mode = time_device_steps(step, steps, warmup, world, eng=eng)
    timing = timing_record(steps)
    value = world * n * steps / (ms * 1e-3)
    ms_k, _ = time_device_steps(step_kernel_only, steps, 1, world, eng=eng)
    k_timing = timing_record(steps)
    g = table.cpu().numpy()
    iters_sum = float(g[:, 5].sum())
    # governing roofline: the fp32 FMA pipe (intensity >> machine balance); the executed-flop rate against the
    # fp32 peak MEASURED in this run, plus the algorithmic I/O rate and the DRAM traffic ncu saw per launch
    peak, peak_src, pk = peaks()
    achieved_io = MPC_BYTES * n * steps / (ms_k * 1e-3) / 1e9
    fpk, fpk_src = fp32_peak(eng)
    tfl = mpc_flops(iters_sum / world, n, T) * steps / (ms_k * 1e-3) / 1e12
    variant = os.environ.get("CRB_MPC_VARIANT", "1")
    kernel = "crb_mpc_tasks_kernel" if variant != "0" else "crb_mpc_solve_kernel"
    traffic = traffic_for("mpc") if n == MPC_N else None
    out = dict(metric="MPC solves/sec (T=20, bicycle model, box-constrained DDP to NLP convergence)",
               value=value, unit="solves/s", ms_per_step=ms / steps, timing=timing,
               config=dict(workload=label or f"mpc_T20_{n}_agents_per_gpu", agents_per_gpu=n,
                           global_agents=n * world, max_iter=MPC_ITER, du_th=MPC_DUTH,
                           max_ls=MPC_LS, stats_allgather="every step, crb_gather_stats inside the graph",
                           l2="3 rotating input sets; per-CTA slab of stage records resident in L2"),
               solver=dict(mean_iters=iters_sum / (world * n),
                           frac_converged=float(g[:, 4].sum()) / (world * n),
                           mean_cost=float(g[:, 0].sum()) / (world * n),
                           checksum=float(g[:, 6].sum())),
               roofline=dict(bound="fp32", achieved=tfl, peak=fpk, unit="TFLOP/s",
                             frac=tfl / fpk, traffic=traffic, peak_source=fpk_src,
                             kernel=kernel, flop_model="executed iterations x (T-1) x (470 + 1.2 x 150) flop, DESIGN.md",
                             solves_per_s_kernel_only=world * n * steps / (ms_k * 1e-3),
                             ms_per_launch=k_timing["ms_per_step"],
                             algorithmic_bytes_per_launch=MPC_BYTES * n,
                             traffic_over_algorithmic=(traffic / (MPC_BYTES * n)) if traffic else None,
                             io_gbs=achieved_io, io_frac_of_hbm=achieved_io / peak))
    # Receding-horizon scheduling (crb_mpc_solve_batched_hinted): the same step with the iteration counts of the previous
    # solve of the same agents as scheduling hints - the long problems start first, which removes most of the tail.
    # The bench repeats one batch, so "previous solve" hints are exact here; the second figure perturbs every hint by
    # a uniform -2..+2 iterations (what a drifting closed loop would hand over).  Same work, same bits (checked).
    if os.environ.get("CRB_MPC_VARIANT", "1") != "0":
        want_iters, want_cost = iters.clone(), cost.clone()
        hint_exact = iters.clone()
        gen = torch.Generator(device="cpu"); gen.manual_seed(1234 + rank)
        hint_noisy = (iters.cpu() + torch.randint(-2, 3, (n,), generator=gen, dtype=torch.int32)).clamp_(min=0).to(dev)
        iters2 = torch.empty_like(iters)
        hinted = {}
        for name, h in (("hints_exact", hint_exact), ("hints_perturbed", hint_noisy)):
            def step_hinted(k, h=h):
                s, xr = sets[k % NSETS]
                eng.mpc_solve_hinted(s, xr, T, h, prm, sol=sol, u0=u0, cost=cost, status=status, iters=iters2)
                eng.stats_reduce(cost, status, iters2, i0=rank * n, out=stats)
                gather_stats(stats, world, eng, out=table)
            ms_h, _ = time_device_steps(step_hinted, steps, 1, world, eng=eng)
            same = bool(torch.equal(iters2, want_iters)) and bool(torch.equal(cost, want_cost))
            hinted[name] = dict(value=world * n * steps / (ms_h * 1e-3), unit="solves/s", ms_per_step=ms_h / steps,
                                speedup_vs_index_order=ms / ms_h, same_bits_as_index_order=same)
        hinted["what"] = ("crb_mpc_solve_batched_hinted: iteration counts of the agents' previous solve as scheduling "
                          "hints (receding-horizon MPC), stats + gather included like the headline step; "
                          "hints_perturbed = every hint off by a uniform -2..+2 iterations")
        out["roofline"]["receding_horizon"] = hinted
    if with_e2e:
        hst, hxr = pinned(st), pinned(xref)
        hsol = torch.empty((nsol, n), dtype=torch.float32).pin_memory()
        hu0 = torch.empty((2, n), dtype=torch.float32).pin_memory()
        hcost = torch.empty(n, dtype=torch.float32).pin_memory()
        hstat = torch.empty(n, dtype=torch.int32).pin_memory()
        hit = torch.empty(n, dtype=torch.int32).pin_memory()
        e_steps = max(2, min(steps, 5))
        ms_e = time_host_steps(lambda k: eng.mpc_solve_host(hst, hxr, T, prm, sol=hsol, u0=hu0, cost=hcost,
                                                            status=hstat, iters=hit), e_steps, 1, world)
        out["e2e"] = dict(value=world * n * e_steps / (ms_e * 1e-3), unit="solves/s",
                          h2d_bytes_per_step=(4 + 4 * T) * 4 * n, d2h_bytes_per_step=(nsol + 5) * 4 * n,
                          path="crb_mpc_solve_batched_host: pinned host inputs / outputs, 8192-problem chunks "
                               "over 8 streams")
    if with_cpu and rank == 0:
        out["cpu_baseline"] = cpu_mpc(st, xref, gpu_u0=u0[:, :MPC_ACC_N].cpu().numpy(),
                                      gpu_cost=cost[:MPC_ACC_N].cpu().numpy())
    return out


MPC_ACC_N = 2048


def _f64_solve(args):
    """Worker of the float64 cross-check (spawned process: numpy only)."""
    from oracle.ref_mpc_f64 import box_ilqr
    st, xr, T = args
    ref = box_ilqr(st.astype(float), xr.reshape(T, 4).T.astype(float), dict(j_tol=0.0, du_th=1e-9, max_iter=200))
    return float(ref["U"][1, 0]), float(ref["U"][0, 0]), float(ref["cost"])


def mpc_accuracy(st, xref, gpu_u0, gpu_cost, T=MPC_T, budget_s=25.0):
    """How far is the binary32 GPU solve (which replaces IPOPT) from the optimum?  The independent float64
    statement (oracle/ref_mpc_f64.py, textbook DDP with np.linalg, converged to du 1e-9) on the first agents of
    the batch, in worker processes; reports max / p99 / median |u0 - u0*| and the relative cost gap."""
    import multiprocessing as mp
    m = min(MPC_ACC_N, st.shape[1], gpu_u0.shape[1])
    jobs = [(st[:, i].copy(), xref[:, i].copy(), T) for i in range(m)]
    res = []
    t0 = time.perf_counter()
    try:
        ctx = mp.get_context("spawn")
        with ctx.Pool(min(32, max(1, host_threads() // 2))) as pool:
            it = pool.imap(_f64_solve, jobs, chunksize=16)
            for r in it:
                res.append(r)
                if time.perf_counter() - t0 > budget_s:
                    pool.terminate()
                    break
    except Exception as exc:   # pragma: no cover
        return dict(error=str(exc))
    k = len(res)
    if k == 0:
        return dict(error="no float64 solves finished in the budget")
    r = np.array(res)
    du = np.maximum(np.abs(r[:, 0] - gpu_u0[0, :k]), np.abs(r[:, 1] - gpu_u0[1, :k]))
    dc = np.abs(r[:, 2] - gpu_cost[:k]) / np.maximum(np.abs(r[:, 2]), 1e-30)
    return dict(sample=k, u0_abs_err_max=float(du.max()), u0_abs_err_p99=float(np.percentile(du, 99)),
                u0_abs_err_median=float(np.median(du)), cost_rel_gap_max=float(dc.max()),
                cost_rel_gap_p99=float(np.percentile(dc, 99)),
                reference="oracle/ref_mpc_f64.py box_ilqr (float64, du_th 1e-9): the KKT point of the reference NLP; "
                          "the reference's own IPOPT solve is capped at 50 ms and unreproducible (mpc:328)",
                seconds=time.perf_counter() - t0)


def cpu_mpc(st=None, xref=None, sample=8192, gpu_u0=None, gpu_cost=None):
    from cpprobotics_b200 import synth
    from oracle import oracle as O
    T = MPC_T
    if st is None:
        course = synth.mpc_course()
        st, pind = synth.mpc_states(sample, course=course)
        xref, _ = synth.mpc_xref_numpy(st, pind, T, course=course)
    st, xref = np.ascontiguousarray(st[:, :sample]), np.ascontiguousarray(xref[:, :sample])
    prm = O.mpc_params(max_iter=MPC_ITER, du_th=MPC_DUTH, max_ls=MPC_LS)
    CPU_SPREAD.clear()
    thr, mask = tuned_threads(lambda c: O.mpc_solve_batched(st, xref, T, prm, nthreads=c))
    v, calls, el = cpu_time(lambda: O.mpc_solve_batched(st, xref, T, prm, nthreads=thr), sample,
                            budget_s=5.0)
    spread = CPU_SPREAD[-1]
    st1, xr1 = np.ascontiguousarray(st[:, :256]), np.ascontiguousarray(xref[:, :256])
    v1, _, _ = cpu_time(lambda: O.mpc_solve_batched(st1, xr1, T, prm, nthreads=1), 256, budget_s=1.0, min_passes=3)
    vb = best_effort(lambda: O.mpc_solve_batched(st, xref, T, prm, nthreads=thr), sample)
    out = dict(value=v, unit="solves/s", cores=thr, kind="port", single_core_value=v1, best_effort_value=vb,
               spread=spread,
               sample=f"median of {calls} passes x {sample} agents (first {sample} of the GPU batch), T={T}, "
                      f"oracle/crb_oracle_mpc.c same algorithm, OpenMP {thr} threads bound to cores (best median of 5 "
                      f"passes at 1/4..1 x the {mask}-cpu mask), {el:.1f} s; "
                      "the reference's CppAD+IPOPT solve cannot be built here (its own budget is "
                      "50 ms per solve, model_predictive_control.cpp:328)")
    if gpu_u0 is not None:
        out["accuracy_vs_float64_optimum"] = mpc_accuracy(st, xref, gpu_u0, gpu_cost)
    return out


def bench_ekf_multistep(eng, rank, world, steps, warmup):
    """Row f-3: 2^20 agents x 100 filter steps per launch, state kept in registers (SURVEY d-3 asks for it).
    16 B/update of (z,u) traffic, so the kernel leaves the HBM roofline and becomes issue-bound."""
    import torch
    from cpprobotics_b200 import synth
    n, ns = 1 << 20, 100
    dev = torch.device("cuda", torch.cuda.current_device())
    x, P, z, u = synth.ekf_inputs(n, i0=rank * n, n_steps=1)
    xd, Pd = torch.from_numpy(x).to(dev), torch.from_numpy(P).to(dev)
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    zd = xd[:2].repeat(ns, 1) + 0.5 * torch.randn((2 * ns, n), device=dev, generator=g)
    ud = torch.tensor([1.0, 0.1], device=dev).repeat(ns).unsqueeze(1) + 0.1 * torch.randn((2 * ns, n), device=dev, generator=g)
    zd, ud = zd.contiguous(), ud.contiguous()
    ms, _ = time_device_steps(lambda k: eng.ekf_estimation(xd, Pd, zd, ud, n_steps=ns), steps, 2, world, eng=eng)
    ok = bool(torch.isfinite(Pd).all().item())
    return dict(metric="EKF updates/sec, 100 steps per launch (state resident in registers)",
                value=world * n * ns * steps / (ms * 1e-3), unit="updates/s", ms_per_step=ms / steps,
                config=dict(workload="ekf_2^20_agents_100_steps_per_launch", finite=ok),
                roofline=dict(bound="hbm", achieved=(16.0 * ns + 160.0) * n * steps / (ms * 1e-3) / 1e9,
                              peak=peaks()[0], unit="GB/s",
                              frac=(16.0 * ns + 160.0) * n * steps / (ms * 1e-3) / 1e9 / peaks()[0], traffic=None,
                              note="16 B/update + 160 B/agent once: far below the HBM roofline by design; the "
                                   "limit here is instruction issue (~460 instructions per update)"))


def copy_ceiling_gbs(nbytes=1 << 30, reps=10):
    """Same-run device copy ceiling (SURVEY d-3): read + write bytes of a 1 GiB torch copy per second."""
    import torch
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    del src, dst
    return 2.0 * nbytes * reps / (ms * 1e-3) / 1e9


def bench_ekf_large(eng, rank, world, steps, warmup):
    """SURVEY d-3 also asks for 16 M agents: the same kernel where the per-launch fixed cost (~1.5 us) is
    amortised over 3.1 GB of traffic."""
    import torch
    from cpprobotics_b200 import synth
    n = 1 << 24
    dev = torch.device("cuda", torch.cuda.current_device())
    x, P, z, u = (torch.from_numpy(a).to(dev) for a in synth.ekf_inputs(1 << 20, i0=rank * n))
    x, P, z, u = (t.repeat(1, 16).contiguous() for t in (x, P, z, u))       # 16 copies of the 2^20 block
    def step(k):
        eng.ekf_estimation(x, P, z, u)
    ms, _ = time_device_steps(step, steps, warmup, world, eng=eng)
    gbs = EKF_BYTES * n * steps / (ms * 1e-3) / 1e9
    return dict(metric="EKF updates/sec, 2^24 agents x 1 step", value=world * n * steps / (ms * 1e-3),
                unit="updates/s", ms_per_step=ms / steps,
                config=dict(workload="ekf_2^24_agents_1_step_per_gpu", l2="3.1 GB per launch >> 126 MB L2"),
                roofline=dict(bound="hbm", achieved=gbs, peak=peaks()[0], unit="GB/s", frac=gbs / peaks()[0],
                              traffic=None, kernel="crb_ekf_step_kernel",
                              algorithmic_bytes_per_launch=EKF_BYTES * n))


def bench_lqr(eng, rank, world, steps, warmup, with_cpu):
    """Row f-4: 2^20 agents, dlqr of lqr_steer_control.cpp (nx=4, nu=1, <=150 DARE iterations each)."""
    import torch
    from cpprobotics_b200 import synth
    n, nx, nu = 1 << 20, 4, 1
    dev = torch.device("cuda", torch.cuda.current_device())
    A, B, Q, R = synth.lqr_inputs(n, nx, i0=rank * n)
    Ad, Bd, Qd, Rd = (torch.from_numpy(a).to(dev) for a in (A, B, Q, R))
    K = torch.empty((nu * nx, n), dtype=torch.float32, device=dev)
    it = torch.empty(n, dtype=torch.int32, device=dev)
    ms, _ = time_device_steps(lambda k: eng.dlqr(Ad, Bd, Qd, Rd, nx, nu, K=K, iters=it), steps, warmup, world,
                              eng=eng)
    mean_it = float(it.float().mean().item())
    flops = mean_it * 2.0 * (5 * 64 + 2 * 16 + 4 + 16) * n * steps    # 5 4x4x4 + 2 4x4x1 + outer + misc per iter
    fpk, fpk_src = fp32_peak(eng)
    out = dict(metric="DARE/LQR gains per second (lqr_steer_control solve_DARE+dlqr, nx=4)",
               value=world * n * steps / (ms * 1e-3), unit="solves/s", ms_per_step=ms / steps,
               config=dict(workload="lqr_dlqr_2^20_agents_per_gpu", mean_dare_iters=mean_it),
               roofline=dict(bound="fp32", achieved=flops / (ms * 1e-3) / 1e12, peak=fpk, unit="TFLOP/s",
                             frac=flops / (ms * 1e-3) / 1e12 / fpk, traffic=None, peak_source=fpk_src,
                             note="no FMA contraction by design (bit-exact with the reference arithmetic): "
                                  "FMUL+FADD pairs, so 0.5 is the ceiling of this fraction",
                             kernel="crb_lqr_dlqr_kernel<4,1>"))
    if with_cpu and rank == 0:
        from oracle import oracle as O
        m = 1 << 16
        thr, mask = tuned_threads(lambda c: O.dlqr_batched(A[:, :m], B[:, :m], Q, R, nx, nu, nthreads=c))
        v, calls, el = cpu_time(lambda: O.dlqr_batched(A[:, :m], B[:, :m], Q, R, nx, nu, nthreads=thr), m, budget_s=3.0)
        out["cpu_baseline"] = dict(value=v, unit="solves/s", cores=thr, kind="port",
                                   sample=f"{calls} x {m} agents, oracle/crb_oracle.c, OpenMP {thr} threads "
                                          f"(fastest of 1/4..1 x the {mask}-cpu mask), {el:.1f} s")
    return out


# sources that define each profiled kernel: profiles/traffic.json carries their hash, so a DRAM-traffic figure
# captured for an older kernel is recognised as stale and NOT reported
KERNEL_SOURCES = {
    "ekf": ["cpprobotics_b200/csrc/crb_ekf.cu", "cpprobotics_b200/csrc/crb_common.cuh"],
    "pf": ["cpprobotics_b200/csrc/crb_pf.cu", "cpprobotics_b200/csrc/crb_common.cuh"],
    "mpc": ["cpprobotics_b200/csrc/crb_mpc_tasks.cu", "cpprobotics_b200/csrc/crb_mpc_core.cuh",
            "cpprobotics_b200/csrc/crb_mpc.cu"],
}


def kernel_stamp(name):
    import hashlib
    h = hashlib.sha256()
    for rel in KERNEL_SOURCES[name]:
        with open(os.path.join(ROOT, rel), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


TRAFFIC_STALE = []


def traffic_for(name):
    """DRAM bytes per launch from the committed ncu --set full capture (profiles/traffic.json), only if the capture
    was taken from the kernel sources this run was built from (hash stamp); otherwise None (and noted)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        rec = json.load(open(p)).get(name)
    except Exception:
        return None
    if isinstance(rec, dict):
        if rec.get("stamp") == kernel_stamp(name):
            return rec.get("bytes")
        TRAFFIC_STALE.append(name)
        return None
    TRAFFIC_STALE.append(name)       # unstamped (round-1 format): cannot be trusted for the current kernel
    return None


# =========================================================================================================
def nest(head, res, key, sub):
    """Copy res[sub][key] (a workload's roofline / e2e / cpu_baseline) under head[key][sub]."""
    if sub in res and key in res[sub] and isinstance(head.get(key), dict):
        head[key][sub.replace("^", "")] = res[sub][key]


def run_ours(args):
    import torch
    from cpprobotics_b200 import Engine
    rank, world, local = dist_setup(args.gpus)
    eng = Engine(local)
    comm_setup(eng, rank, world)
    res = {}
    cpu = (not args.no_cpu) and world == 1     # cpu_baseline: rank 0 at N = 1 only (the contract)
    restore = (lambda: None)
    if cpu:
        restore, pin_note = cpu_pin_one_numa_node()
    with ClockSampler(local) as clk:
        head = bench_ekf(eng, rank, world, args.steps, args.warmup, with_cpu=cpu, dump_dir=args.dump_outputs)
        if args.workload in ("all", "pf"):
            res["pf"] = bench_pf(eng, rank, world, args.steps, args.warmup, with_cpu=cpu)
        if args.workload in ("all", "pf"):
            res["pf_full_iteration"] = bench_pf_iteration(eng, rank, world, 10, 3)
        if args.workload in ("all", "ekf100"):
            res["ekf_100_steps"] = bench_ekf_multistep(eng, rank, world, 3, 2)
        if args.workload in ("all", "ekf16m"):
            res["ekf_16M_agents"] = bench_ekf_large(eng, rank, world, 5, 3)
        if args.workload in ("all", "lqr"):
            res["lqr"] = bench_lqr(eng, rank, world, max(3, args.steps // 5), 3, with_cpu=cpu)
        if args.workload in ("all", "mpc"):
            # BASELINE configs[3]: 65 536 agents per GPU (weak scaling like the headline)
            res["mpc"] = bench_mpc(eng, rank, world, max(3, args.steps // 5), max(1, args.warmup // 3),
                                   with_cpu=cpu)
            # BASELINE configs[4] AS WRITTEN: 2^20 agents in total, sharded over the N GPUs (strong scaling:
            # 2^20 / N per GPU), index-addressed shards, one all-gather of the cost statistics per call
            tot = 1 << 20
            res["mpc_config5"] = bench_mpc(eng, rank, world, 3, 1, with_cpu=False, n=tot // world,
                                           label=f"mpc_T20_2^20_agents_sharded_over_{world}_gpus "
                                                 f"({tot // world} per GPU; BASELINE.json configs[4])",
                                           with_e2e=(world == 1))
            c5 = res["mpc_config5"]
            c5["config"]["scaling"] = "strong (total fixed at 2^20)"
            c5["per_gpu_solves_per_s"] = c5["value"] / world
            c5["roofline"]["frac_of_n_gpus_peak"] = c5["roofline"]["frac"]     # per-GPU flop rate / per-GPU peak
    restore()
    cfg = {"workload": "ekf_2^20_agents_1_step_per_gpu (BASELINE.json configs[1])",
           "agents_per_gpu": EKF_N, "global_agents": EKF_N * world,
           "l2": "3 rotating buffer sets, 303 MB of inputs > 126 MB L2",
           "collective": "one all-gather of 8 doubles per rank (libcrb crb_gather_stats, NCCL) inside the captured "
                         "graph, once per replay of K steps",
           "launch": head["launch_mode"], "timing": head["timing"]}
    line = {
        "metric": "EKF updates/sec (4-state/2-obs predict+update, batched)",
        "value": head["value"], "unit": "updates/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": head["ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "clocks": clk.summary(), "e2e": head["e2e"], "gpu_launches": head["launches"],
        "roofline": head["roofline"],
    }
    if "cpu_baseline" in head:
        line["cpu_baseline"] = head["cpu_baseline"]
        line["cpu_baseline"]["pinning"] = pin_note
    # BASELINE.json's metric is "EKF updates/sec & MPC solves/sec ...": the MPC (and PF) figures of this run are part
    # of the record the driver parses, not an appendix
    for sub in ("mpc", "pf", "mpc_config5"):
        for key in ("roofline", "e2e", "cpu_baseline"):
            nest(line, res, key, sub)
    if "mpc" in res:
        cfg["mpc_solves_per_s"] = res["mpc"]["value"]
        cfg["mpc_workload"] = res["mpc"]["config"]["workload"] + " (BASELINE.json configs[3])"
        cfg["mpc_ms_per_step"] = res["mpc"]["ms_per_step"]
        cfg["mpc_solver"] = res["mpc"]["solver"]
        if "accuracy_vs_float64_optimum" in res["mpc"].get("cpu_baseline", {}):
            cfg["mpc_accuracy_vs_float64_optimum"] = res["mpc"]["cpu_baseline"]["accuracy_vs_float64_optimum"]
    if "mpc" in res and "receding_horizon" in res["mpc"]["roofline"]:
        rh = res["mpc"]["roofline"]["receding_horizon"]
        cfg["mpc_solves_per_s_with_iteration_hints"] = {k: rh[k]["value"] for k in ("hints_exact", "hints_perturbed")}
    if "mpc_config5" in res:
        c5 = res["mpc_config5"]
        cfg["mpc_config5"] = dict(workload=c5["config"]["workload"], solves_per_s=c5["value"],
                                  per_gpu_solves_per_s=c5["per_gpu_solves_per_s"], ms_per_step=c5["ms_per_step"],
                                  frac_of_fp32_peak=c5["roofline"]["frac"], n_gpus=world)
        if "receding_horizon" in c5["roofline"]:
            cfg["mpc_config5"]["solves_per_s_with_iteration_hints"] = {
                k: c5["roofline"]["receding_horizon"][k]["value"] for k in ("hints_exact", "hints_perturbed")}
    if "pf" in res:
        cfg["pf_particles_per_s"] = res["pf"]["value"]
        cfg["pf_workload"] = res["pf"]["config"]["workload"] + " (BASELINE.json configs[2])"
    if TRAFFIC_STALE:
        cfg["traffic_stale"] = sorted(set(TRAFFIC_STALE))
    ni = NUMA_INFO.get(local, {})
    cfg["host_buffers_numa"] = {"node_of_gpu": ni.get("node"), "unknown_because": ni.get("why")}
    if res:
        line["extra"] = res
    if rank == 0:
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores (the oracle port: the real
    Eigen / CppAD / IPOPT sources cannot be built in this image).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    restore, pin_note = cpu_pin_one_numa_node()
    from oracle import oracle as O
    from cpprobotics_b200 import synth
    n = EKF_N
    x, P, z, u = synth.ekf_inputs(n)
    thr, mask = tuned_threads(lambda c: O.ekf_step_batched(x, P, z, u, nthreads=c, inplace=True))
    for _ in range(args.warmup):
        O.ekf_step_batched(x, P, z, u, nthreads=thr, inplace=True)
    ts = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        O.ekf_step_batched(x, P, z, u, nthreads=thr, inplace=True)
        ts.append(time.perf_counter() - t0)
    ts = np.array(ts)
    el = float(ts.sum())
    v = n * args.steps / el
    vb = best_effort(lambda: O.ekf_step_batched(x, P, z, u, nthreads=thr, inplace=True), n)
    line = {
        "impl": "reference", "metric": "EKF updates/sec (4-state/2-obs predict+update, batched)",
        "value": v, "unit": "updates/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ekf_2^20_agents_1_step_per_gpu (BASELINE.json configs[1])",
                   "agents_per_gpu": EKF_N},
        "cpu_baseline": {"value": v, "unit": "updates/s", "cores": thr, "kind": "port", "best_effort_value": vb,
                         "pinning": pin_note,
                         "spread": dict(passes=int(ts.size), fastest=n / ts.min(), slowest=n / ts.max(),
                                        median=n / float(np.median(ts))),
                         "sample": f"{args.steps} x {n} agents x 1 step per timed step, oracle/crb_oracle.c "
                                   f"(-O2 -ffp-contract=off), OpenMP {thr} threads bound to cores (best median of 5 "
                                   f"passes at 1/4..1 x the {mask}-cpu mask)"},
        "e2e": {"value": v, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.workload in ("all", "pf"):
        line["cpu_baseline"]["pf"] = cpu_pf()
    if args.workload in ("all", "mpc"):
        line["cpu_baseline"]["mpc"] = cpu_mpc()
        line["config"]["mpc_solves_per_s"] = line["cpu_baseline"]["mpc"]["value"]
    restore()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "ekf", "ekf100", "ekf16m", "pf", "mpc", "lqr"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
