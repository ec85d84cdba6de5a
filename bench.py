#!/usr/bin/env python
"""bench.py — atom-grid evaluations/s (energy + force) of the GridForce path on B200.

    python bench.py --gpus 1 --steps K --warmup W                 # this repo's CUDA path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                          # the reference's own CPU kernel, all host cores

Workload (config.workload): BASELINE.json configs[4] — 65,536 ligand replicas x 47 atoms x 3 grids of 192^3.
  N = 1   the whole batch on one GPU.
  N > 1   STRONG scaling (default, what configs[4] names): the 65,536 replicas are block-partitioned over the N ranks
          (shard_bounds), grids replicated, no collective on the force path, and ONE gather of the per-replica energies
          after the last step, inside the timed region. --scaling weak gives every rank 65,536 replicas instead.
A "step" = one evaluation of the whole batch: positions -> per-replica energies + forces for every atom on every grid,
one kernel launch per GPU. Successive steps evaluate DIFFERENT pose sets (2N sets of the shard size rotate), so that the
bytes touched between two uses of the same data are the same at every N and exceed L2.

  value      device-resident inputs; K steps per window, W_n windows, CUDA events on the launching stream around each
             window, max over ranks per window, median over windows. The K-step loop (+ the final gather) is a CUDA graph
             whose launches carry programmatic-dependent-launch edges (small launches — a rank's shard at N >= 4 — then
             run the tile-striding instantiation of the kernel); the same loop with direct launches and without launch
             overlap is timed in the same run and reported under "variants".
  e2e        the same through the plugin's batched entry point GridForceBatch (pinned HOST positions in, energies + FP32
             forces out; H2D/D2H inside the timed region); FP64 forces, energy-only and the bare C ABI beside it.
  roofline   algorithmic bytes per evaluation (DESIGN.md: 36 + 52/G bytes, G grids per atom) x evaluations per launch /
             average launch duration, against the measured HBM copy bandwidth in MEASURED_PEAKS.json
The data path of an N > 1 run is the C ABI only (gfb_comm_*: the energy gather as one flag-in-data kernel over the NVLink
peer mappings by default — push + wait, the fused tail of the last launch and ncclAllGather selectable — and a device-side
rendezvous of the ranks in front of each timed window);
torch.distributed is the launcher's bootstrap channel (NCCL id, IPC handles), the barrier and the max over ranks.
Only the cpu_baseline leg and --impl reference load anything from oracle/ (the test-only CPU oracle); the cpu_baseline
leg also uses it to CHECK a sample of the timed kernel's output — a mismatch refuses the JSON line.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "atom-grid evals/s (E+F)"
UNIT = "evals/s"
REPLICAS_TOTAL = 65536
REPLICAS_PER_GPU = REPLICAS_TOTAL          # weak scaling, and N = 1
N_ATOMS = 47
N_GRIDS = 3
GRID_N = 192
# device-side start rendezvous of the timed windows (N > 1). The held kernel waits for a host write that follows the
# enqueue of the window, so it is off when launches block the host (CUDA_LAUNCH_BLOCKING=1 would wait for the 20 s timeout).
RENDEZVOUS = (os.environ.get("GFB_BENCH_RENDEZVOUS", "1") != "0" and os.environ.get("CUDA_LAUNCH_BLOCKING", "0") in ("", "0"))
KERNEL_SOURCES = ("gf_eval_lines.cuh", "gf_eval_lines_f64.cuh", "gf_gather.cuh", "gf_kernels.cuh", "gf_params.h", "gf_launch_lines.cu")


def b_alg(n_grids, precision=0, forces=True):
    """Algorithmic bytes per atom-grid evaluation (SURVEY.md §8d / DESIGN.md §4): stencil + scaling factor + (position +
    force accumulate + order) / G. Energy-only evaluations do not touch the 24 force bytes."""
    per_atom = 52.0 if forces else 28.0
    return (36.0 + per_atom / n_grids) if precision == 0 else (72.0 + per_atom / n_grids)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def kernel_source_hash():
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        h.update(open(os.path.join(ROOT, "openmmgridforce_b200", "csrc", name), "rb").read())
    return h.hexdigest()[:16]


def physical_roofline(traffic, traffic_src, launch_us, peak_gbs):
    """The same launch against the roofline with the DRAM bytes ncu MEASURED for it instead of the algorithmic bytes: how
    close the kernel runs to the HBM peak given the traffic it really causes (whole sectors fetched for 32-byte stencils
    raise it above the algorithmic bytes, L2 hits lower it). None when no valid capture is committed."""
    if not traffic or "LOWER BOUND" in (traffic_src or ""):
        return None
    ach = traffic / (launch_us * 1e-6) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs,
            "bytes": "dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu), / this run's launch time"}


def measured_traffic(workload_key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/r2_traffic.json,
    written by tools/ncu_traffic.py) — reported only while the kernel sources still hash to what was profiled."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(path):
        return None, "no ncu capture committed for this round"
    doc = json.load(open(path))
    entry = doc.get(workload_key)
    if not entry:
        return None, f"profiles/r2_traffic.json has no entry for {workload_key}"
    if entry.get("source_sha256_16") != kernel_source_hash():
        return None, "kernel sources changed since the ncu capture in profiles/r2_traffic.json"
    return float(entry["dram_bytes_per_launch"]), entry.get("source", "profiles/r2_traffic.json")


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 100 ms from just before the timed device loop until the last
    GPU measurement of the run (device loop, e2e loop, and at N=1 the C3/C4 loops)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.tmp,
                                         stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.tmp.flush()
        rows = [r.split(",") for r in open(self.tmp.name).read().splitlines() if r.count(",") >= 8]
        os.unlink(self.tmp.name)
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in rows:
            for name, v in zip(names, r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=float(rows[0][2]), reasons=sorted(reasons), samples=len(rows))
        return out


def bind_to_gpu_cpus(gpu_index):
    """Restrict this process to the CPU cores NVML reports as local to the GPU (what `nvidia-smi topo -m` prints), so that
    its pinned buffers are allocated on that NUMA node. Returns a short description for the JSON line; never fatal."""
    if os.environ.get("GFB_BIND_CPUS", "1") == "0":
        return "off"
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus ({min(cpus)}-{max(cpus)})"
        return "no local cpus reported"
    except Exception as exc:
        return f"unavailable ({type(exc).__name__})"


def pinned_array(shape, dtype=np.float64):
    """numpy view over page-locked host memory (torch is the allocator; no torch type crosses the C ABI)."""
    import torch
    t = torch.empty(tuple(shape), dtype={np.float64: torch.float64, np.float32: torch.float32, np.int64: torch.int64}[dtype],
                    pin_memory=True)
    return t.numpy(), t


def workload_config(n_gpus, scaling="strong"):
    """The workload both arms (this repo's and --impl reference) run. Nothing arm-specific in here."""
    strong = scaling == "strong" or n_gpus == 1
    total = REPLICAS_TOTAL if strong else REPLICAS_PER_GPU * n_gpus
    return {"workload": f"configs[4]: {total} ligand replicas x {N_ATOMS} atoms x {N_GRIDS} grids of {GRID_N}^3"
                        + (f", sharded over {n_gpus} GPUs" if n_gpus > 1 else " on one GPU"),
            "replicas_total": total, "replicas_per_gpu": total // n_gpus, "atoms_per_replica": N_ATOMS,
            "grids": N_GRIDS, "grid_points": [GRID_N] * 3, "precision": "mixed", "scaling": "strong" if strong else "weak",
            "parallelism": f"replica-sharded x{n_gpus}",
            "evals_per_step": total * N_ATOMS * N_GRIDS}


def pose_sets(W, rank, world, strong, n_sets):
    """This rank's pose sets. Set 0 is its block of the canonical batch (replicas [lo, hi) of the 65,536 generated from
    SEED, or — weak scaling — a 65,536-replica batch of its own); the other sets are the same number of replicas drawn
    with other seeds. Returns (workload of set 0, [pos arrays], (lo, hi))."""
    from openmmgridforce_b200.sharding import shard_bounds
    if strong:
        lo, hi = shard_bounds(REPLICAS_TOTAL, world, rank)
        w = W.c5_sharded_replicas(n_replicas=REPLICAS_TOTAL, n=GRID_N, replica_offset=lo, n_local=hi - lo)
    else:
        lo, hi = rank * REPLICAS_PER_GPU, (rank + 1) * REPLICAS_PER_GPU
        w = W.c5_sharded_replicas(n_replicas=REPLICAS_PER_GPU, n=GRID_N, pose_seed=W.SEED + rank)
    half = 0.5 * w.spacing[0] * (GRID_N - 1)
    sets = [w.pos]
    for j in range(1, n_sets):
        sets.append(W.ligand_replicas(hi - lo, (half, half, half), seed=W.SEED + 7919 * j + rank, escape_shift=(0.9, 0.0, 0.0)))
    return w, sets, (lo, hi)


# ----------------------------------------------------------------------------------------------------------------
# device-timed loops
# ----------------------------------------------------------------------------------------------------------------
class DeviceLoop:
    """Device-resident pose sets + per-set fixed-point force buffers + rotating energy accumulators, and the K-step window
    that is timed: K evaluation launches on `stream`, the last of which carries (or is followed by) the energy gather."""

    def __init__(self, torch, gf, dev, kern, sets, n_atoms, stream, comm=None, gather_mode="none", lo=0, total=0,
                 force_mode=None):
        self.torch, self.gf, self.dev, self.kern, self.stream, self.comm = torch, gf, dev, kern, stream, comm
        self.gather_mode = gather_mode
        tdev = torch.device("cuda", dev.ordinal)
        self.r, self.a = sets[0].shape[0], n_atoms
        n = self.r * self.a
        self.stride = ((n + 31) // 32) * 32
        self.force_mode = gf.FORCE_FIXED_ADD if force_mode is None else force_mode
        self.d_pos = [torch.from_numpy(np.ascontiguousarray(p)).to(tdev) for p in sets]
        if self.force_mode == gf.FORCE_FIXED_ADD:
            self.d_f = [torch.zeros(3 * self.stride, dtype=torch.int64, device=tdev) for _ in sets]
        elif self.force_mode == gf.FORCE_F32_STORE:
            self.d_f = [torch.zeros(3 * n, dtype=torch.float32, device=tdev) for _ in sets]
        elif self.force_mode < 0:
            self.d_f = [None for _ in sets]
        else:
            self.d_f = [torch.zeros(3 * n, dtype=torch.float64, device=tdev) for _ in sets]
        self.d_e = [torch.zeros(self.r, dtype=torch.float64, device=tdev) for _ in range(3)]
        self.lo, self.total = lo, total
        self.d_gathered = torch.zeros(max(total, 1), dtype=torch.float64, device=tdev)
        self.set_evals = [0] * len(sets)      # evaluations accumulated into each set's force buffer
        self.last = None                      # (set index, accumulator index) of the most recent step
        torch.cuda.synchronize()

    @staticmethod
    def accumulators(steps):
        """Which of the three accumulators step j adds into: consecutive steps differ, and the last differs from the
        first (whose buffer it clears for the next window). Step j's launch clears a[j + 1] (a[steps] = a[0])."""
        a = [j % 3 for j in range(steps)]
        if steps > 1 and a[-1] == a[0]:
            a[-1] = next(x for x in (1, 2) if x != a[-2])
        return a

    def window(self, first, steps, count=True):
        gf, kern, s = self.gf, self.kern, self.stream.cuda_stream
        acc = self.accumulators(steps)
        for j in range(steps):
            si = (first + j) % len(self.d_pos)
            e = self.d_e[acc[j]]
            nxt = self.d_e[acc[(j + 1) % steps]] if steps > 1 else None
            f = self.d_f[si].data_ptr() if self.d_f[si] is not None else None
            last = j == steps - 1
            if steps == 1:
                e.zero_()
            if last and self.gather_mode == "fused":
                kern.execute_device_gather(self.comm, self.lo, self.r, self.a, self.d_pos[si].data_ptr(), e.data_ptr(), f,
                                           max(self.force_mode, 0), self.stride, s, d_energies_clear=nxt.data_ptr() if nxt is not None else None)
                self.comm.gather_wait(self.d_gathered.data_ptr(), s)
            else:
                kern.execute_device(self.r, self.a, self.d_pos[si].data_ptr(), e.data_ptr(), None, f, max(self.force_mode, 0),
                                    self.stride, None, s, d_energies_clear=nxt.data_ptr() if nxt is not None else None)
                if last and self.gather_mode == "nccl":
                    self.comm.all_gather(e.data_ptr(), self.d_gathered.data_ptr(), self.r, s)
                elif last and self.gather_mode == "push":
                    self.comm.gather_push(e.data_ptr(), self.r, self.lo, s)
                    self.comm.gather_wait(self.d_gathered.data_ptr(), s)
                elif last and self.gather_mode == "ll":
                    self.comm.gather(e.data_ptr(), self.r, self.lo, self.d_gathered.data_ptr(), s)
            if count:
                self.set_evals[si] += 1
            self.last = (si, acc[j])

    def time_windows(self, steps, warmup, windows, pdl, graph, barrier=None, reduce_max=None):
        """Returns per-window milliseconds (max over ranks when reduce_max is given) and the launches per window; the steps
        evaluated inside the timed windows are counted in self.timed_steps."""
        torch, gf = self.torch, self.gf
        self.kern.set_launch_overlap(pdl)
        n_sets = len(self.d_pos)
        self.timed_steps = 0
        with torch.cuda.stream(self.stream):
            done = 0
            while done < warmup:                      # untimed warm-up steps, in windows of at most K
                k = min(steps, warmup - done)
                self.window(done, k)
                done += k
            self.stream.synchronize()
            g = None
            if graph and steps > 1:
                gf.Graph.begin(self.dev, self.stream.cuda_stream)
                self.window(0, steps, count=False)
                g = gf.Graph.end(self.dev, self.stream.cuda_stream)
                g.launch(self.stream.cuda_stream)             # untimed first replay (graph upload)
                self._count_replay(0, steps)
                self.stream.synchronize()
            out = []
            for w in range(windows):
                first = (w * steps) % n_sets if g is None else 0
                if barrier is not None:
                    barrier()
                # N > 1: the host barrier lets the ranks go tens of microseconds apart, and the window's one collective
                # (the energy gather) would be charged that skew. A device-side rendezvous in front of the first event
                # starts all ranks within an NVLink round trip; it is held until this rank's window has been enqueued.
                rendezvous = self.comm is not None and barrier is not None and RENDEZVOUS
                if rendezvous:
                    self.comm.rendezvous(self.stream.cuda_stream, hold=True)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                evals_before = sum(self.set_evals)
                e0.record(self.stream)
                if g is not None:
                    g.launch(self.stream.cuda_stream)
                    self._count_replay(0, steps)
                else:
                    self.window(first, steps)
                e1.record(self.stream)
                if rendezvous:
                    self.comm.rendezvous_release()
                self.stream.synchronize()
                self.timed_steps += sum(self.set_evals) - evals_before
                if barrier is not None:
                    barrier()
                out.append(e0.elapsed_time(e1))
            if g is not None:
                g.close()
        self.kern.set_launch_overlap(False)
        if reduce_max is not None:
            out = reduce_max(out)
        launches = steps + {"fused": 1, "push": 2, "ll": 1}.get(self.gather_mode, 0)
        return out, launches

    def _count_replay(self, first, steps):
        acc = self.accumulators(steps)
        for j in range(steps):
            self.set_evals[(first + j) % len(self.d_pos)] += 1
        self.last = ((first + steps - 1) % len(self.d_pos), acc[-1])

    def last_step_results(self, n_sample):
        """(positions, energies, forces per evaluation) of the first n_sample replicas of the set the most recent step
        evaluated — what the timed kernel left in its buffers."""
        torch, gf = self.torch, self.gf
        si, ai = self.last
        n = min(n_sample, self.r)
        en = self.d_e[ai][:n].cpu().numpy()
        pos = self.d_pos[si][:n].cpu().numpy()
        tdev = self.d_pos[si].device
        na = self.r * self.a
        if self.force_mode == gf.FORCE_FIXED_ADD:
            d_out = torch.empty(na, 3, dtype=torch.float64, device=tdev)
            self.dev.fixed_to_f64(self.d_f[si].data_ptr(), self.stride, na, d_out.data_ptr(), self.stream.cuda_stream)
            self.stream.synchronize()
            f = d_out.view(self.r, self.a, 3)[:n].cpu().numpy() / float(self.set_evals[si])
        else:
            f = None
        return pos, en, f


def summarize(ms_windows, steps):
    s = sorted(ms_windows)
    med = s[len(s) // 2]
    return {"ms_per_step": med / steps, "min_ms_per_step": s[0] / steps, "max_ms_per_step": s[-1] / steps, "windows": len(s)}


VARIANTS = (("pdl+graph", True, True), ("pdl", True, False), ("graph", False, True), ("plain", False, False))


def run_variants(loop, steps, warmup, windows, barrier=None, reduce_max=None, which=VARIANTS):
    out = {}
    launches = 0
    for name, pdl, graph in which:
        ms, launches = loop.time_windows(steps, warmup, windows, pdl, graph, barrier, reduce_max)
        out[name] = summarize(ms, steps)
    return out, launches


def time_e2e(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    return time.perf_counter() - t0


def grid_forces_for(gfp, w):
    """The workload as a script would hand it to the plugin: one GridForce per grid (bulk setters)."""
    forces = []
    for g in range(w.n_grids):
        f = gfp.GridForce()
        f.addGridCounts(*w.counts)
        f.addGridSpacing(*w.spacing)
        f.setGridOrigin(*w.origin)
        f.setGridValues(w.grids[g])
        f.setScalingFactors(w.scaling[g])
        f.setOutOfBoundsRestraint(w.oob_k[g])
        f.setForceGroup(g)
        forces.append(f)
    return forces


def run_e2e(gf, kern, w, local_rank, steps, reduce_max_scalar=None, barrier=None):
    """End to end through the plugin's batched entry point (GridForceBatch, pointer overloads on pinned caller buffers)
    and, for comparison, through the bare C ABI. Every call returns with the results in host memory."""
    import openmmgridforce_b200.gridforceplugin as gfp
    r = w.n_replicas
    pos_h, _k1 = pinned_array(w.pos.shape)
    pos_h[...] = w.pos
    f64_h, _k2 = pinned_array(w.pos.shape)
    f32_h, _k3 = pinned_array(w.pos.shape, np.float32)
    e_h, _k4 = pinned_array((r,))
    batch = gfp.GridForceBatch(local_rank, "mixed")
    for f in grid_forces_for(gfp, w):
        batch.addForce(f)
    calls = {
        "GridForceBatch::evaluateWithForcesF32": lambda: batch.evaluateWithForcesF32(pos_h, r, e_h, f32_h),
        "GridForceBatch::evaluateWithForces": lambda: batch.evaluateWithForces(pos_h, r, e_h, f64_h),
        "GridForceBatch::evaluate (energy only)": lambda: batch.evaluate(pos_h, r, e_h),
        "gfb_kernel_execute_host (C ABI, FP64 forces)": lambda: kern.execute_host(pos_h, forces=f64_h, energies_out=e_h),
    }
    d2h = {"GridForceBatch::evaluateWithForcesF32": w.pos.nbytes // 2 + 8 * r, "GridForceBatch::evaluateWithForces": w.pos.nbytes + 8 * r,
           "GridForceBatch::evaluate (energy only)": 8 * r, "gfb_kernel_execute_host (C ABI, FP64 forces)": w.pos.nbytes + 8 * r}
    out = {}
    for name, fn in calls.items():
        if barrier is not None:
            barrier()
        secs = time_e2e(fn, steps, 3)
        if reduce_max_scalar is not None:
            secs = reduce_max_scalar(secs)
        out[name] = {"ms_per_step": secs / steps * 1e3, "timed_steps": steps, "h2d_bytes_per_step": int(w.pos.nbytes),
                     "d2h_bytes_per_step": int(d2h[name])}
    # the energies the batched entry point returned last (energy-only call ran third, C ABI last): keep them for the check
    batch.evaluateWithForcesF32(pos_h, r, e_h, f32_h)
    result = (e_h.copy(), f32_h.copy())
    batch.close()
    return out, result


def run_single_ligand(gf, dev, steps):
    """configs[1]: one 47-atom ligand in three 208x278x231 grids, one evaluation per MD step through the host API
    (positions in, energy + forces out, synchronous). OpenMM's integrator is not available here, so the figure is the
    grid-force-limited upper bound: steps/s x 4 fs (example/input.json:24)."""
    from openmmgridforce_b200 import workloads as W
    w = W.c2_single_ligand()
    grids = [gf.Grid(dev, w.counts, w.spacing, w.origin, v, gf.PRECISION_MIXED) for v in w.grids]
    kern = gf.Kernel(dev, grids, w.scaling, oob_k=w.oob_k)
    pos_h, _t1 = pinned_array(w.pos.shape)
    pos_h[...] = w.pos
    f_h, _t2 = pinned_array(w.pos.shape)
    e_h, _t3 = pinned_array((1,))
    secs = time_e2e(lambda: kern.execute_host(pos_h, forces=f_h, energies_out=e_h), steps, 50)
    e_launch, f_launch = float(e_h[0]), f_h.copy()
    # The same calls with the resident evaluator (gfb_kernel_set_resident): a block stays on the GPU between steps, no
    # launch and no synchronise per step.
    kern.set_resident(True)
    # A tool that serialises kernel launches (ncu, compute-sanitizer) makes every resident step wait for the block's idle
    # time-out: probe a few steps first and leave the measurement out instead of spending minutes on it.
    probe = time_e2e(lambda: kern.execute_host(pos_h, forces=f_h, energies_out=e_h), 3, 2) / 3
    serialised = probe > 5e-3
    if serialised:
        resident = {"skipped": f"a resident step took {probe * 1e3:.1f} ms: kernel launches are being serialised (profiler?)"}
    else:
        rsecs = time_e2e(lambda: kern.execute_host(pos_h, forces=f_h, energies_out=e_h), steps, 50)
        resident = {"us_per_step": rsecs / steps * 1e6, "steps_per_s": steps / rsecs, "block_launches": kern.resident_launches(),
                    "gpu_us_last_step": dict(zip(("evaluation", "results_issued"), (float(v) for v in kern.resident_timeline()))),
                    "same_result_as_launch_path": bool(abs(float(e_h[0]) - e_launch) <= 1e-6 * abs(e_launch) and
                                                       np.abs(f_h - f_launch).max() <= 1e-5 * np.abs(f_launch).max()),
                    "api": "gfb_kernel_execute_host after gfb_kernel_set_resident(1), ctypes loop"}
    kern.close()
    for g in grids:
        g.close()
    sps = steps / secs
    # The same step as an OpenMM integrator would issue it: System with three GridForce objects on the B200 platform
    # plugin (libOpenMMGridForceB200.so), Context::calcForcesAndEnergy timed from C++. The platform evaluates the three
    # forces of a step in ONE launch (step fusion, DESIGN.md §4.5).
    plugin = None
    try:
        import openmmgridforce_b200.gridforceplugin as gfp
        system = gfp.System()
        for _ in range(w.n_atoms):
            system.addParticle(1.0)
        for f in grid_forces_for(gfp, w):
            system.addForce(f)
        for key, props in (("launch", None), ("resident", {"ResidentKernel": "true"})):
            if key == "resident" and serialised:
                plugin["resident_kernel"] = {"skipped": "kernel launches are being serialised (profiler?)"}
                continue
            ctx = gfp.Context(system, gfp.Platform.getPlatformByName("B200"), props)
            ctx.setPositions(w.pos.reshape(-1, 3))
            ctx.timeEvaluations(200)
            psecs, _e = ctx.timeEvaluations(steps)
            entry = {"us_per_step": psecs * 1e6, "steps_per_s": 1.0 / psecs, "grid_force_limited_ns_per_day": 4e-6 * 86400.0 / psecs,
                     "energy": _e}
            if key == "launch":
                plugin = dict(entry, api="B200 platform plugin: Context::calcForcesAndEnergy over 3 GridForces, C++ step loop")
            else:
                plugin["resident_kernel"] = dict(entry, api='the same Context created with {"ResidentKernel": "true"}')
            del ctx
    except Exception as exc:      # reported, not fatal: the C-ABI figure above stands on its own
        plugin = dict(plugin or {}, error=repr(exc))
    return {"workload": w.name, "us_per_step": secs / steps * 1e6, "steps_per_s": sps, "openmm_plugin_path": plugin,
            "resident_evaluator": resident,
            "grid_force_limited_ns_per_day": sps * 4e-6 * 86400.0, "value": w.evals * sps, "unit": UNIT,
            "note": "latency-bound: one launch per step on host-mapped memory + one synchronize; upper bound on MD ns/day at 4 fs"}


def run_other_workload(torch, gf, dev, stream, name, steps, warmup, windows, peak_gbs, l2_gbs):
    """C3 / C4 (and C5 in DOUBLE precision / energy only) device-resident on one GPU, rotating sets, the same window
    machinery; FIXED_ADD unless the name says otherwise."""
    from openmmgridforce_b200 import workloads as W
    precision, force_mode, forces = gf.PRECISION_MIXED, gf.FORCE_FIXED_ADD, True
    if name == "C3":
        w = W.c3_million_atoms()
        rng = np.random.default_rng(99)
        length = w.spacing[0] * (w.counts[0] - 1)
        sets = [w.pos] + [rng.uniform(0.0, 0.999 * length, size=w.pos.shape) for _ in range(7)]
    elif name == "C4":
        w = W.c4_batched_replicas()
        sets = [w.pos] + [W.ligand_replicas(w.n_replicas, W.ligand47()[0].mean(axis=0), seed=W.SEED + 10 + i,
                                            escape_shift=(1.0, 0.0, 0.0)) for i in range(15)]
    else:      # C5 variants on the resident grids' workload
        w, sets, _ = pose_sets(W, 0, 1, True, 2)
        if name == "C5_double":
            precision = gf.PRECISION_DOUBLE
        elif name == "C5_energy_only":
            force_mode, forces = -1, False
    # interpolation methods 1 and 2 on their record layouts (a stencil = two 128-byte records instead of one 32-byte slot)
    layout = {"C5_bspline": gf.LAYOUT_BSPLINE, "C5_tricubic": gf.LAYOUT_HERMITE}.get(name)
    grids = [gf.Grid(dev, w.counts, w.spacing, w.origin, v, precision, layout=layout) for v in w.grids]
    kern = gf.Kernel(dev, grids, w.scaling, oob_k=w.oob_k)
    loop = DeviceLoop(torch, gf, dev, kern, sets, w.n_atoms, stream, force_mode=force_mode)
    variants, _ = run_variants(loop, steps, warmup, windows, which=(VARIANTS[0], VARIANTS[3]))
    best = variants["pdl+graph"]
    rate = w.evals / (best["ms_per_step"] * 1e-3)
    bpe = b_alg(w.n_grids, 1 if precision == gf.PRECISION_DOUBLE else 0, forces)
    if layout is not None:
        bpe += 256.0 - 32.0      # two 128-byte records per evaluation in place of the 32-byte trilinear stencil
    ach = rate * bpe / 1e9
    traffic, traffic_src = measured_traffic(name)
    suffix = {"C5_double": " (DOUBLE precision)", "C5_energy_only": " (energy only)",
              "C5_bspline": " (cubic B-spline, interpolation method 1, BSPLINE records)",
              "C5_tricubic": " (tricubic Hermite, interpolation method 2, HERMITE records)"}.get(name, "")
    out = {"workload": w.name + suffix,
           "value": rate, "unit": UNIT, "us_per_step": best["ms_per_step"] * 1e3,
           "us_per_step_no_overlap_direct_launches": variants["plain"]["ms_per_step"] * 1e3,
           "eval_path": kern.eval_path(),
           "l2": f"rotating {len(sets)} position/force sets (aggregate footprint > L2)",
           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs,
                        "traffic": traffic, "traffic_source": traffic_src, "bytes_per_eval": bpe},
           "roofline_l2_gather": {"achieved": ach, "peak": l2_gbs, "unit": "GB/s", "frac": ach / l2_gbs if l2_gbs else None},
           "roofline_measured_traffic": physical_roofline(traffic, traffic_src, best["ms_per_step"] * 1e3, peak_gbs)}
    if ach > peak_gbs:
        out["roofline"]["note"] = ("above 1: the algorithmic bytes count every stencil record as a DRAM read, and L2 serves part of "
                                   "them (the poses cluster around the grid centre); see roofline_measured_traffic")
    if name in ("C3", "C4"):
        pos_h, _t1 = pinned_array(w.pos.shape)
        pos_h[...] = w.pos
        f_h, _t2 = pinned_array(w.pos.shape, np.float32)
        e_h, _t3 = pinned_array((w.n_replicas,))
        secs = time_e2e(lambda: kern.execute_host(pos_h, forces=f_h, force_mode=gf.FORCE_F32_STORE, energies_out=e_h), steps, 3)
        out["e2e"] = {"value": w.evals * steps / secs, "unit": UNIT, "h2d_bytes_per_step": int(w.pos.nbytes),
                      "d2h_bytes_per_step": int(w.pos.nbytes // 2 + 8 * w.n_replicas), "api": "gfb_kernel_execute_host, FP32 forces"}
    del loop
    kern.close()
    for g in grids:
        g.close()
    return out


# ----------------------------------------------------------------------------------------------------------------
# CPU legs (the only users of oracle/)
# ----------------------------------------------------------------------------------------------------------------
def _cpu_oracle_for_sample(bindings, w, pos):
    """One Context holding the sample's atoms (replicas flattened), G GridForces — evaluated by the reference's own
    kernel when oracle/_ref is present, else by the C restatement."""
    n_sample = pos.shape[0]
    n = n_sample * w.n_atoms
    flat = np.ascontiguousarray(pos.reshape(n, 3))
    scaling = np.tile(w.scaling, (1, n_sample))
    if bindings.ref_available():
        ref = bindings.RefOracle(n, w.counts, w.spacing, w.origin, w.grids, scaling, oob_k=w.oob_k)
        return "reference", (lambda reps: ref.execute_repeat(flat, reps)), n * w.n_grids
    port = bindings.PortOracle(w.counts, w.spacing, w.origin, w.grids, scaling, oob_k=w.oob_k)

    def run(reps):
        for _ in range(reps):
            for g in range(w.n_grids):
                port.execute(flat, g)
    return "port", run, n * w.n_grids


def cpu_baseline(w, target_seconds=12.0, n_sample=2048, check=None):
    """Single-threaded (the reference is single-threaded as written) on a bounded sample of the same workload. With
    `check` = [(label, positions, energies, forces or None), ...] the oracle also CHECKS what the timed GPU paths
    produced: per replica |E - E_ref| <= max(1e-6 |E_ref|, 6e-8 sum|s v|), forces 1e-5 relative (max-norm)."""
    from oracle import bindings
    from openmmgridforce_b200 import workloads as W
    checked = []
    for label, pos, en, f in (check or []):
        port = bindings.PortOracle(w.counts, w.spacing, w.origin, w.grids, w.scaling, oob_k=w.oob_k)
        ge_ref, f_ref = port.execute_batched(np.ascontiguousarray(pos), n_threads=os.cpu_count() or 1)
        e_ref = ge_ref.sum(axis=1)
        bound = np.maximum(1e-6 * np.abs(e_ref), 6e-8 * W.mixed_energy_bound(w, pos))
        bad_e = np.abs(en - e_ref) > bound
        msg = None
        if bad_e.any():
            i = int(np.argmax(np.abs(en - e_ref) / np.maximum(bound, 1e-300)))
            msg = f"{label}: energy of replica {i} is {en[i]!r}, the oracle says {e_ref[i]!r} (bound {bound[i]:.3e})"
        if msg is None and f is not None:
            err = np.abs(f - f_ref).max() / np.abs(f_ref).max()
            if not err <= 1e-5:
                msg = f"{label}: forces differ from the oracle by {err:.3e} relative (max-norm)"
        if msg:
            raise SystemExit("bench.py: the timed path's output failed the oracle check — " + msg)
        checked.append({"what": label, "replicas": int(pos.shape[0]), "max_energy_err_over_bound": float((np.abs(en - e_ref) / np.maximum(bound, 1e-300)).max()),
                        "force_rel_err": float(np.abs(f - f_ref).max() / np.abs(f_ref).max()) if f is not None else None})
    n_sample = min(n_sample, w.n_replicas)
    kind, run, evals = _cpu_oracle_for_sample(bindings, w, w.pos[:n_sample])
    run(3)                                      # warm-up (also gets the reference's debug prints out of the way)
    t0 = time.perf_counter()
    run(2)
    per = (time.perf_counter() - t0) / 2
    reps = max(3, int(target_seconds / max(per, 1e-6)))
    t0 = time.perf_counter()
    run(reps)
    secs = time.perf_counter() - t0
    return {"value": evals * reps / secs, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": f"first {n_sample} replicas ({n_sample * w.n_atoms} atoms x {w.n_grids} grids), {reps} passes, {secs:.1f} s",
            "output_check": checked}


def reference_arm(args):
    """The reference's own CPU implementation on all host threads, on the SAME workload as the repo arm: the 65,536
    replicas are cut into one contiguous block per host thread (one reference Context per thread, as example/sampler.py
    keeps one per replica), and a step is ONE pass of every thread over its block = the whole batch once."""
    from oracle import bindings
    from openmmgridforce_b200 import workloads as W
    from openmmgridforce_b200.sharding import shard_bounds
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    cfg = workload_config(args.gpus, args.scaling)
    passes = max(1, cfg["replicas_total"] // REPLICAS_TOTAL)      # weak scaling at N > 1: the 65,536 poses N times per step
    total = REPLICAS_TOTAL
    if os.environ.get("GFB_REF_REPLICAS"):            # bounded sample for slow hosts; the JSON line then says so
        total = min(total, int(os.environ["GFB_REF_REPLICAS"]))
    w = W.c5_sharded_replicas(n_replicas=REPLICAS_TOTAL, n=GRID_N, n_local=total)
    runs, kind = [], "port"
    for t in range(threads):
        lo, hi = shard_bounds(total, threads, t)
        if hi == lo:
            continue
        kind, run, _ = _cpu_oracle_for_sample(bindings, w, w.pos[lo:hi])
        runs.append(run)
    evals_per_step = total * passes * w.n_atoms * w.n_grids
    runs[0](3)                                  # serial warm-up: the reference's static debug counters are not thread-safe

    def one_step():
        th = [threading.Thread(target=r, args=(passes,)) for r in runs]
        for t in th:
            t.start()
        for t in th:
            t.join()

    for _ in range(args.warmup):
        one_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_step()
    secs = time.perf_counter() - t0
    value = evals_per_step * args.steps / secs
    sample = (f"{len(runs)} host threads x {total // max(len(runs), 1)} replicas x {w.n_atoms} atoms x {w.n_grids} grids = "
              f"{total} replicas, {passes} pass(es) per step (ctypes releases the GIL; one reference Context per thread)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": cfg["scaling"],
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": len(runs), "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="K: the steps of every timed window (the headline times --windows windows of K steps; the other "
                         "variants, the other workloads and the per-call e2e loops time K steps or calls each)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default=os.environ.get("GFB_BENCH_SCALING", "strong"), choices=["strong", "weak"],
                    help="N>1: strong = the named config (65,536 replicas in total, sharded); weak = 65,536 per GPU")
    ap.add_argument("--energy-gather", default=os.environ.get("GFB_ENERGY_GATHER", "ll"), choices=["ll", "push", "fused", "nccl"],
                    help="N>1: the one gather of per-replica energies after the last step — ll: ONE kernel of this library "
                         "behind the last launch, flag-in-data packets over the NVLink peer mappings (publish + wait + copy-out, "
                         "no fence, no flag round; default); push: peer stores + arrival flags by one kernel, wait + copy-out "
                         "by a second; fused: the push from the tail of the last evaluation launch; nccl: ncclAllGather. The "
                         "result is checked against another method outside the timed region.")
    ap.add_argument("--windows", type=int, default=5, help="timed K-step windows (median reported)")
    ap.add_argument("--no-extras", action="store_true", help="skip C2/C3/C4/C5 variants and the CPU baseline (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR (N=1 only): energies.npy [replicas] float64 and "
                         "forces.npy [replicas, atoms, 3] float32, 37.5 MB in all; the inputs are seeded, so two builds run "
                         "with the same arguments can be compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    args.windows = max(args.windows, 1)
    if args.dump_outputs and (args.gpus != 1 or args.impl != "b200"):
        raise SystemExit("--dump-outputs needs --gpus 1 and --impl b200")

    if args.impl == "reference":
        reference_arm(args)
        return

    # stdout carries ONE JSON line; anything libraries print while the run sets up (NCCL's version banner) goes to stderr
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import openmmgridforce_b200 as gf
    from openmmgridforce_b200 import workloads as W

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    strong = args.scaling == "strong" or world == 1
    torch.cuda.set_device(local_rank)
    tdev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_cpus(local_rank)     # pinned host buffers are then first-touched on the GPU's own NUMA node
    dev = gf.Device(local_rank)             # raises if the CUDA library or an sm_100 GPU is missing: no fallback
    stream = torch.cuda.Stream(device=tdev)
    peak_gbs, peak_src = measured_peaks()

    # ---- launcher-side plumbing (N > 1): torch.distributed carries the NCCL id and the IPC handles, the barrier and
    #      the max over ranks; the energy gather itself is gfb_comm_* ----------------------------------------------------
    dist, comm = None, None
    barrier = reduce_max = reduce_max_scalar = None
    n_sets = 2 * world if strong else 2
    w, sets, (lo, hi) = pose_sets(W, rank, world, strong, n_sets)
    total = REPLICAS_TOTAL if strong else REPLICAS_PER_GPU * world
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=tdev)
        uid = [gf.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = gf.Comm(dev, world, rank, uid[0])
        handles = [None] * world
        dist.all_gather_object(handles, comm.gather_alloc(total))
        comm.gather_attach(handles)

        def barrier():
            dist.barrier()
            torch.cuda.synchronize()

        def reduce_max(ms_list):
            t = torch.tensor(ms_list, dtype=torch.float64, device=tdev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.tolist()

        def reduce_max_scalar(x):
            return reduce_max([x])[0]

    grids = [gf.Grid(dev, w.counts, w.spacing, w.origin, v, gf.PRECISION_MIXED) for v in w.grids]
    kern = gf.Kernel(dev, grids, w.scaling, oob_k=w.oob_k)
    gather_mode = args.energy_gather if world > 1 else "none"
    loop = DeviceLoop(torch, gf, dev, kern, sets, N_ATOMS, stream, comm=comm, gather_mode=gather_mode, lo=lo, total=total)

    l2_gbs = dev.bench_sector_gather(32 << 20, 1 << 24, 10) if rank == 0 else 0.0
    if barrier is not None:
        barrier()
    host_copy = dev.bench_host_copy(64 << 20, 5)        # every rank at the same time: the share each GPU gets
    sampler = ClockSampler(local_rank)
    if barrier is not None:
        barrier()
    torch.cuda.synchronize()
    sampler.start()

    head_name = "pdl+graph" if args.steps > 1 else "pdl"
    variants, launches = run_variants(loop, args.steps, args.warmup, args.windows, barrier, reduce_max,
                                      which=[v for v in VARIANTS if v[0] == head_name])
    headline = variants[head_name]
    timed_steps = loop.timed_steps
    gather_check = None
    if world > 1:
        comm.gather_status()
        # the gathered energies of the last window must equal the OTHER gather method's result on the same accumulators
        si, ai = loop.last
        other = torch.zeros(total, dtype=torch.float64, device=tdev)
        if gather_mode in ("fused", "push", "ll"):
            comm.all_gather(loop.d_e[ai].data_ptr(), other.data_ptr(), loop.r, stream.cuda_stream)
        else:
            dist.all_gather_into_tensor(other, loop.d_e[ai])
        torch.cuda.synchronize()
        if not torch.equal(other, loop.d_gathered):
            raise SystemExit(f"rank {rank}: energy gather ({gather_mode}) does not match the reference all-gather")
        gather_check = f"{gather_mode} gather == " + ("ncclAllGather via gfb_comm_all_gather" if gather_mode != "nccl" else "torch all_gather_into_tensor") + " (bit-identical, outside the timed region)"
    dev_sample = loop.last_step_results(1024)
    # taken now (the later windows overwrite the buffers), written to disk after the last measurement
    dump = loop.last_step_results(loop.r)[1:] if args.dump_outputs else None
    # this rank's own per-step time (not the max over ranks, no gather) for the roofline of ITS kernel
    saved_mode, loop.gather_mode = loop.gather_mode, "none"
    own_ms, _ = loop.time_windows(args.steps, 0, 3, True, args.steps > 1)
    kernel_us = sorted(own_ms)[1] / args.steps * 1e3
    # the same loop launched the other ways (direct launches, no launch overlap): reported, not the headline
    loop.gather_mode = saved_mode
    others, _ = run_variants(loop, args.steps, 0, max(3, args.windows // 2), barrier, reduce_max,
                             which=[v for v in VARIANTS if v[0] != head_name])
    variants.update(others)

    weak = None
    if world > 1 and strong and os.environ.get("GFB_BENCH_WEAK", "1") != "0":
        # the weak-scaling curve as a second figure: every rank evaluates 65,536 replicas of its own (no gather change)
        w_weak, sets_weak, _ = pose_sets(W, rank, world, False, 2)
        comm_w_total = REPLICAS_PER_GPU * world
        loop_w = DeviceLoop(torch, gf, dev, kern, sets_weak, N_ATOMS, stream, comm=None, gather_mode="none", lo=0, total=0)
        vw, _ = run_variants(loop_w, args.steps, 4, 3, barrier, reduce_max, which=(VARIANTS[0],))
        weak = {"scaling": "weak", "replicas_total": comm_w_total, "ms_per_step": vw["pdl+graph"]["ms_per_step"],
                "value": comm_w_total * N_ATOMS * N_GRIDS / (vw["pdl+graph"]["ms_per_step"] * 1e-3), "unit": UNIT,
                "note": "65,536 replicas per GPU, no energy gather in this window"}
        del loop_w

    # ---- end to end --------------------------------------------------------------------------------------------------
    e2e, e2e_result = run_e2e(gf, kern, w, local_rank, args.steps, reduce_max_scalar, barrier)
    if barrier is not None:
        barrier()
    host_copy_after = dev.bench_host_copy(64 << 20, 5)

    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        for name in ("C3", "C4", "C5_double", "C5_energy_only", "C5_bspline", "C5_tricubic"):
            extras[name] = run_other_workload(torch, gf, dev, stream, name, args.steps, args.warmup, 3, peak_gbs, l2_gbs)
        extras["C2"] = run_single_ligand(gf, dev, args.steps)
    clocks = sampler.stop()

    evals_step_rank = w.n_replicas * N_ATOMS * N_GRIDS
    evals_step = total * N_ATOMS * N_GRIDS
    value = evals_step / (headline["ms_per_step"] * 1e-3)
    ach = evals_step_rank * b_alg(N_GRIDS) / (kernel_us * 1e-6) / 1e9
    host_copy_all = [list(host_copy)]
    if world > 1:
        t = torch.tensor(list(host_copy) + list(host_copy_after), dtype=torch.float64, device=tdev)
        allt = torch.empty(world * 6, dtype=torch.float64, device=tdev)
        dist.all_gather_into_tensor(allt, t)
        host_copy_all = allt.view(world, 6).tolist()

    if rank == 0:
        cfg = workload_config(world, args.scaling)
        head_api = "GridForceBatch::evaluateWithForcesF32"
        traffic, traffic_src = measured_traffic("C5" if world == 1 else f"C5_shard_{world}")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": headline["ms_per_step"], "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
                "dtype": "f32 interpolation, f64 index/energy, i64 fixed-point forces", "data": "synthetic", "config": cfg,
                "run": {"windows": headline["windows"], "timed_steps": timed_steps, "min_ms_per_step": headline["min_ms_per_step"],
                        "max_ms_per_step": headline["max_ms_per_step"],
                        "launch": ("CUDA graph of the K-step loop; launches carry programmatic-dependent-launch edges (a step's "
                                   "blocks fetch positions/records and issue their force atomics during the previous step's "
                                   "tail, and wait for it before their energy writes)" if args.steps > 1 else "direct launches, PDL")
                                  + ("; launches of at most 6 tiles per resident block (N >= 4 here) run the tile-striding "
                                     "instantiation of the same kernel (DESIGN.md 4.1)" if world > 1 else ""),
                        "start_rendezvous": ("device-side rendezvous of all ranks (gfb_comm_rendezvous) between the host barrier and "
                                             "the window's first event" if (world > 1 and RENDEZVOUS) else None),
                        "pose_sets": f"{n_sets} sets of {w.n_replicas} replicas rotate (inputs larger than L2 between re-uses; no L2 flush)",
                        "energy_gather": gather_mode if world > 1 else "none (one GPU)",
                        "energy_gather_when": "once per window, after the last step, inside the timed region" if world > 1 else "n/a",
                        "gather_check": gather_check,
                        "data_path": "C ABI only (gfb_kernel_execute_device[_gather], gfb_comm_*, gfb_graph_*); torch.distributed = bootstrap, barrier, max over ranks"},
                "variants": {k: {"ms_per_step": v["ms_per_step"], "value": evals_step / (v["ms_per_step"] * 1e-3)} for k, v in variants.items()},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs,
                             "traffic": traffic, "traffic_unit": "bytes per launch", "traffic_source": traffic_src,
                             "peak_source": peak_src, "kernel": "gf_eval_lines_kernel<3 grids, FIXED_ADD> (one 128-byte record per cell)",
                             "bytes_per_eval": b_alg(N_GRIDS), "evals_per_launch": evals_step_rank, "launch_us": kernel_us},
                "roofline_l2_gather": {"achieved": ach, "peak": l2_gbs, "unit": "GB/s", "frac": ach / l2_gbs if l2_gbs else None,
                                       "peak_source": "gfb_bench_sector_gather: random 32-byte sectors over 32 MB, this run"},
                "roofline_measured_traffic": physical_roofline(traffic, traffic_src, kernel_us, peak_gbs),
                "e2e": {"value": evals_step / (e2e[head_api]["ms_per_step"] * 1e-3), "unit": UNIT,
                        "h2d_bytes_per_step": e2e[head_api]["h2d_bytes_per_step"], "d2h_bytes_per_step": e2e[head_api]["d2h_bytes_per_step"],
                        "ms_per_step": e2e[head_api]["ms_per_step"],
                        "api": head_api + " (plugin batched entry point, pointer overloads on pinned caller buffers: positions uploaded by the "
                               "copy engine in 8 chunks, FP32 forces stored by the kernels straight into the caller's buffer); per rank on its shard, max over ranks",
                        "variants": {k: dict(v, value=evals_step / (v["ms_per_step"] * 1e-3)) for k, v in e2e.items()},
                        "host_copy_gbs": {"per_rank_h2d_d2h_both_before_and_after": host_copy_all,
                                          "note": "gfb_bench_host_copy, 64 MB pinned, every rank at the same time: the PCIe/host-memory share each GPU gets",
                                          "h2d_floor_ms_per_step": w.pos.nbytes / (min(r[0] for r in host_copy_all) * 1e9) * 1e3}},
                "gpu_launches": int(launches * args.windows), "clocks": clocks, "cpu_binding": numa}
        if ach > peak_gbs:
            line["roofline"]["note"] = ("above 1: the denominator is the measured COPY bandwidth (equal read and write streams); this "
                                        "launch's DRAM traffic is 80 % reads (roofline_measured_traffic: ncu's bytes for the same "
                                        "launch over this run's launch time), and the HBM3e interface is nominally 7.7 TB/s")
        if weak is not None:
            line["weak_scaling"] = weak
        if world == 1 and not args.no_extras:
            line["other_workloads"] = extras
            checks = [("device loop, last timed step (FIXED_ADD, PDL + graph)",) + dev_sample,
                      ("GridForceBatch::evaluateWithForcesF32", w.pos[:1024], e2e_result[0][:1024], e2e_result[1][:1024].astype(np.float64))]
            line["cpu_baseline"] = cpu_baseline(w, check=checks)
        if dump is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "energies.npy"), dump[0])
            np.save(os.path.join(args.dump_outputs, "forces.npy"), dump[1].astype(np.float32))
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        comm.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
