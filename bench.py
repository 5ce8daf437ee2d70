#!/usr/bin/env python
"""bench.py -- EM/VBEM iterations per second on BASELINE.json configs[1] (headline), plus Stage A
(selective-alignment Mreads/s at human-transcriptome scale, configs[2] shape) in the "stage_a" object.

Workload (config 2, the largest EM-only configuration; fits one GPU): synth_eq(seed=1):
500 000 equivalence classes over 250 000 transcripts (nnz ~3.0 M, sum of counts ~20 M),
VBEM (salmon's default), 1000 forced iterations per step (min_iter = max_iter = 1000).

A "step" = one CollapsedEMOptimizer::optimize-equivalent run of 1000 iterations.
  value : iterations / s with the class table resident in HBM (sb_em_run only),
  e2e   : the same through sb_em_optimize with HOST buffers (pinned): H2D of the CSR
          table + device-side preparation (combined weights, both layouts) + 1000
          iterations + D2H of alpha, all inside the timed region.
L2 is flushed (512 MB memset) before every timed step; inside a step the working set
(~75 MB) is L2-resident by nature of the workload (the same table is swept 1000x).

N > 1 (torchrun, one rank per GPU): weak scaling -- every rank holds its OWN 500k-class
table (the eq-classes of its read shard) and alpha is all-reduced once per iteration.
value = N x (iterations / s): 500k-class-shard iterations per second.

--impl reference : the CPU path (oracle port, OpenMP over all host cores) on the same
workload; each step is a bounded sample of iterations.

--dump-outputs DIR : after the timed steps, what the last timed step of each path returned to its caller, as
DIR/<name>.npy in float64 (see collect_outputs); the inputs are seeded, so two builds can be compared array by array.

The bench writes nothing into the source tree (it may be read-only): what it compiles or caches goes to temp dirs.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True


def _bind_rank_to_cores():
    """Host-side placement, decided BEFORE libgomp is loaded.

    One process (N=1): OpenMP threads pinned to cores (close).  Under torchrun (N>1) every rank gets its OWN
    contiguous slice of the host cores -- the slice of the cores NVML reports as near its GPU when that is
    available, else an equal share -- and OMP_NUM_THREADS = a bounded part of it.  (Round 1 exported
    OMP_PROC_BIND=close / OMP_PLACES=cores together with torchrun's OMP_NUM_THREADS=1, which made libgomp bind
    every rank's launch thread to place 0: all ranks on one core.  VERDICT r1 weak #4.)"""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    try:
        avail = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return None
    if world <= 1:
        os.environ.setdefault("OMP_PROC_BIND", "close")
        os.environ.setdefault("OMP_PLACES", "cores")
        return avail
    for k in ("OMP_PROC_BIND", "OMP_PLACES", "GOMP_CPU_AFFINITY"):
        os.environ.pop(k, None)
    lw = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    near = None
    try:
        import pynvml
        pynvml.nvmlInit()
        n_gpu = pynvml.nvmlDeviceGetCount()
        words = (max(avail) // 64) + 1
        sets = []
        for g in range(n_gpu):
            h = pynvml.nvmlDeviceGetHandleByIndex(g)
            m = pynvml.nvmlDeviceGetCpuAffinity(h, words)
            sets.append(tuple(c for c in avail if (m[c // 64] >> (c % 64)) & 1))
        mine = sets[local]
        sharers = [g for g in range(min(lw, n_gpu)) if sets[g] == mine]
        if mine and local in sharers:
            k = len(mine) // len(sharers)
            i = sharers.index(local)
            near = list(mine[i * k:(i + 1) * k]) if k > 0 else None
    except Exception:  # noqa: BLE001
        near = None
    if not near:
        k = max(1, len(avail) // lw)
        near = avail[local * k:(local + 1) * k] or avail
    os.sched_setaffinity(0, near)
    os.environ["OMP_NUM_THREADS"] = str(max(1, min(16, len(near))))
    return near


_AFFINITY = _bind_rank_to_cores()

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

C2 = dict(C=500_000, M=250_000, total_count=20_000_000)
ITERS_PER_STEP = 1000


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes_per_iter(eq, vbem=True):
    """SURVEY.md section 8d: nnz*(4+8) + C*(8+8) + M*(8+8+8) [+ M*16 for VBEM's expTheta]."""
    return eq.nnz * 12 + eq.n_classes * 16 + eq.n_txps * 24 + (eq.n_txps * 16 if vbem else 0)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.t_mark = index, None, [], None

    def mark(self):
        """start of the timed region: samples that arrive from now on are 'timed', earlier ones 'warm-up'"""
        self.t_mark = time.perf_counter()

    def wait_first(self, timeout=4.0):
        """nvidia-smi needs a moment to start: block until its first line is in (so that short timed regions get samples)"""
        t0 = time.perf_counter()
        while self.proc and not self.lines and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        timed = [ln for (t, ln) in self.lines if self.t_mark is None or t >= self.t_mark]
        window = "timed region"
        if len(timed) < 3:      # a timed region shorter than a few sampling periods: add the warm-up steps (same kernels, same load)
            timed = [ln for (_, ln) in self.lines]
            window = "warm-up + timed region (timed region shorter than 3 sampling periods)"
        for ln in timed:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # samples under load = upper half of the observed clocks
        hi = sorted(sm)[len(sm) // 2:]
        return {"sm_mhz": statistics.median(hi), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


_CPU_BEST = {}
CPU_PROBE_FILE = os.path.join(tempfile.gettempdir(), f"salmon_b200_cpu_probe_{os.getuid()}.json")     # per box and user
CPU_REPEATS = 5
_SCRATCH = None


def scratch_dir():
    """a temporary directory for this run (removed at exit): host helpers the bench compiles go there"""
    global _SCRATCH
    if _SCRATCH is None:
        _SCRATCH = tempfile.TemporaryDirectory(prefix="sb_bench_")
    return _SCRATCH.name


def _cpu_probe_load():
    try:
        d = json.load(open(CPU_PROBE_FILE))
        if d.get("host_cores") == (os.cpu_count() or 1):
            return d
    except Exception:  # noqa: BLE001
        pass
    return {"host_cores": os.cpu_count() or 1}


def cpu_port_rate(eq, proj, eff, uniq, vbem, budget_s, threads):
    """Times the CPU port (oracle) on a bounded number of iterations.

    The port mirrors the reference's decomposition (parallel_for over classes + CAS f64 adds).  On many-core
    hosts that decomposition is contention-bound, so the thread count is chosen ONCE per box by a probe over
    {all, 64, 32, 16, 8} cores and the serial restatement (median of three differences per candidate); the
    choice is written to CPU_PROBE_FILE and reused by every later call on that box (a reference-arm run and a
    B200-arm run on the same box time the same thread count).  Threads are pinned
    (OMP_PROC_BIND=close, OMP_PLACES=cores, set before libgomp loads).  The reported rate is the MEDIAN of
    CPU_REPEATS timed runs; returns (rate, iterations per run, threads, [rates])."""
    import oracle_lib as O
    from salmon_b200 import default_params

    def run(n, t):
        p = default_params(use_vbem=vbem, min_iter=n, max_iter=n)
        t0 = time.perf_counter()
        if t == 0:
            O.em_optimize(eq, proj, eff, uniq, p)
        else:
            O.em_optimize(eq, proj, eff, uniq, p, mt=True, n_threads=t)
        return time.perf_counter() - t0

    def per_iter(t):
        run(2, t)                      # warm-up (thread pool, page faults)
        d, a = [], None
        for _ in range(3):
            a, b = run(4, t), run(16, t)    # fixed serial setup cancels in the difference
            d.append((b - a) / 12.0)
        return max(statistics.median(d), 1e-6), a

    key = f"em:{eq.n_classes}:{eq.nnz}:{int(bool(vbem))}:{threads}"
    if key not in _CPU_BEST:
        cache = _cpu_probe_load()
        if key in cache:
            _CPU_BEST[key] = tuple(cache[key])
        else:
            cands = sorted({t for t in (threads, 64, 32, 16, 8) if 0 < t <= threads}, reverse=True) + [0]
            best = None
            for t in cands:
                pi, a = per_iter(t)
                if best is None or pi < best[1]:
                    best = (t, pi, a)
            _CPU_BEST[key] = best
            cache[key] = list(best)
            try:
                json.dump(cache, open(CPU_PROBE_FILE, "w"))
            except Exception:  # noqa: BLE001
                pass
    t, pi, a = _CPU_BEST[key]
    n = int(max(20, min(ITERS_PER_STEP, budget_s / CPU_REPEATS / pi)))
    setup = max(a - 4 * pi, 0.0)
    run(2, t)
    rates = [n / max(run(n, t) - setup, 1e-9) for _ in range(CPU_REPEATS)]
    return statistics.median(rates), n, (t if t else 1), rates


# --------------------------------------------------------------------------------------------
# Stage A: selective alignment + online assignment + eq-class builder (BASELINE.json configs[2] shape)
# --------------------------------------------------------------------------------------------
SA = dict(n_genes=60_000, reads_per_step=2_097_152, batch=262_144, read_len=100)


def stage_a_algorithmic_bytes(n_frags, read_len, c, band=15):
    """SURVEY.md section 8d: B_frag = 2*len/4 + L*96 + E/4 + P*8 + A*(len+2*band)/4 + 32*K (+ 4*sum|label|)."""
    return (n_frags * 2 * read_len / 4 + c["lookups"] * 96 + c["postings"] * 8 + c["candidates"] * (read_len + 2 * band) / 4
            + 32 * c["kept"] + 4 * c["label_entries"])


def stage_a_traffic(frags_per_launch):
    """DRAM bytes per seed-kernel launch from the committed ncu --set full capture (per fragment x fragments per launch)"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic_r2.json")))["stage_a"]
        return t["dram_bytes_per_fragment"] * frags_per_launch
    except Exception:  # noqa: BLE001
        return None


def stage_a_workload(rank, small=False):
    from salmon_b200.synth import synth_txome, synth_reads_fast, flatten_txome
    g = SA["n_genes"] // (20 if small else 1)
    txps, _ = synth_txome(seed=44, n_genes=g)
    flat = flatten_txome(txps)
    left, right, _ = synth_reads_fast(txps, seed=7 + rank, n=SA["reads_per_step"] // (16 if small else 1),
                                      read_len=SA["read_len"], flat=flat)
    return txps, flat, left, right


def write_fastq_pair(dirname, left, right):
    """the step's reads as two plain 4-line FASTQ files (vectorised writer): what `sb_salmon quant -1 -2` would be given"""
    lut = np.frombuffer(b"ACGTN", dtype=np.uint8)
    paths = []
    for tag, codes in (("1", left), ("2", right)):
        n, L = codes.shape
        rec = np.empty((n, 3 + L + 3 + L + 1), dtype=np.uint8)
        rec[:, 0:3] = np.frombuffer(b"@r\n", dtype=np.uint8)
        rec[:, 3:3 + L] = lut[codes]
        rec[:, 3 + L:6 + L] = np.frombuffer(b"\n+\n", dtype=np.uint8)
        rec[:, 6 + L:6 + 2 * L] = ord("I")
        rec[:, 6 + 2 * L] = 10
        path = os.path.join(dirname, f"bench_{tag}.fq")
        rec.tofile(path)
        paths.append(path)
    return paths


_GZ_PARSER_SNIPPET = r"""
import sys, time, numpy as np
sys.path.insert(0, sys.argv[1])
from salmon_b200 import _capi
g1, g2, batch, L, threads, k = sys.argv[2], sys.argv[3], int(sys.argv[4]), int(sys.argv[5]), int(sys.argv[6]), int(sys.argv[7])
bufs = (np.empty((batch, L), np.uint8), np.empty((batch, L), np.uint8), np.empty(batch, np.uint32), np.empty(batch, np.uint32))
best = 0.0
for _ in range(2):
    rf = _capi.ReadFiles(g1, g2, n_threads=threads)
    t0 = time.perf_counter(); tot = 0
    while True:
        got = rf.next_batch(batch, L, out=bufs)[0]
        if got == 0:
            break
        tot += got
    dt = time.perf_counter() - t0
    rf.close()
    assert tot == k, (tot, k)
    best = max(best, tot / dt / 1e6)
print("PARSER_RATE", best)
"""


def stage_a_from_gz(idx, d, f1, f2, n, L, batch, threads, max_pairs=1_000_000):
    """The first max_pairs records of the two FASTQ files through `gzip -1`; the parser alone, then the whole
    `sb_salmon quant` command on the .gz files.  Both run as CHILD PROCESSES with a time limit: the parallel inflater is
    the newest host code of the path, and an extra measurement must never be able to hang the bench line.  idx None
    (CPU-only check of this function): the parser rate alone."""
    import re
    import subprocess
    k = min(n, max_pairs)
    rec = 2 * L + 7
    gz = [p + ".gz" for p in (f1, f2)]
    procs = []
    for src, dst in zip((f1, f2), gz):
        fo = open(dst, "wb")
        ph = subprocess.Popen(["head", "-c", str(k * rec), src], stdout=subprocess.PIPE)
        pg = subprocess.Popen(["gzip", "-1"], stdin=ph.stdout, stdout=fo)
        ph.stdout.close()
        procs.append((ph, pg, fo))
    for ph, pg, fo in procs:
        pg.wait(timeout=300); ph.wait(timeout=60); fo.close()
        if pg.returncode != 0:
            raise RuntimeError("gzip failed")
    out = {"files": "the first %d pairs, gzip -1" % k, "pairs": int(k), "parser_threads": threads,
           "gz_bytes": int(sum(os.path.getsize(g) for g in gz))}
    r = subprocess.run([sys.executable, "-B", "-c", _GZ_PARSER_SNIPPET, ROOT, gz[0], gz[1], str(batch), str(L), str(threads), str(k)],
                       capture_output=True, text=True, timeout=180)
    m = re.search(r"PARSER_RATE ([0-9.eE+-]+)", r.stdout)
    if r.returncode != 0 or not m:
        raise RuntimeError("parser child failed: " + (r.stderr or r.stdout)[-300:])
    out["parser_only_mreads_s"] = float(m.group(1))
    if idx is not None:
        ipath = os.path.join(d, "idx")
        os.makedirs(ipath, exist_ok=True)
        idx.save(os.path.join(ipath, "sb_index.bin"))
        exe = os.path.join(ROOT, "salmon_b200", "sb_salmon")
        cmd = [exe, "quant", "-i", ipath, "-l", "IU", "-1", gz[0], "-2", gz[1], "-o", os.path.join(d, "out_gz"), "-p", str(threads),
               "--batch", str(batch), "--maxReadLen", str(L)]
        best = None
        for _ in range(2):
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
            m = re.search(r"mapping ([0-9.]+) s \(([0-9.]+) ms on the device, ([0-9.]+) M fragments/s end to end", r.stderr)
            m2 = re.search(r"(\d+) fragments observed, (\d+) mapped", r.stderr)
            if r.returncode != 0 or not m or not m2:
                raise RuntimeError("sb_salmon quant on the .gz files failed: " + r.stderr[-300:])
            cur = {"files_to_classes_mreads_s": float(m.group(3)), "map_seconds": float(m.group(1)), "map_device_ms": float(m.group(2)),
                   "n_mapped": int(m2.group(2))}
            m3 = re.search(r"mapping set-up ([0-9.]+) s", r.stderr)
            if m3:
                cur["map_setup_ms"] = float(m3.group(1)) * 1e3
                cur["files_to_classes_streaming_mreads_s"] = k / max(cur["map_seconds"] - float(m3.group(1)), 1e-9) / 1e6
            if int(m2.group(1)) != k:
                raise RuntimeError(f"sb_salmon observed {m2.group(1)} of {k} pairs")
            if best is None or cur["files_to_classes_mreads_s"] > best["files_to_classes_mreads_s"]:
                best = cur
        out.update(best)
        out["api"] = "sb_salmon quant (child process; map_seconds includes sb_map_create)"
    return out


def stage_a_from_files(idx, left, right, batch, ncores):
    """row f1 measured: FASTQ files -> parser threads -> length buckets (pinned) -> sb_map_batch -> classes -> EM, through
    sb_quant_files (the C++ driver `sb_salmon quant` calls); and the parser alone (sb_reads_next into host buffers)."""
    import shutil
    import tempfile
    from salmon_b200 import _capi
    need = 2 * left.shape[0] * (2 * left.shape[1] + 7) + (64 << 20)
    base = None
    if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK):
        sv = os.statvfs("/dev/shm")
        if sv.f_bavail * sv.f_frsize > need:
            base = "/dev/shm"
    d = tempfile.mkdtemp(prefix="sb_bench_", dir=base)
    try:
        n, L = left.shape
        f1, f2 = write_fastq_pair(d, left, right)
        threads = max(1, min(32, ncores - 2))
        out = {"files": "2 plain FASTQ files in " + (base or "the temp dir"), "pairs": int(n), "parser_threads": threads}
        bufs = (np.empty((batch, L), np.uint8), np.empty((batch, L), np.uint8), np.empty(batch, np.uint32), np.empty(batch, np.uint32))
        best = 0.0
        for _ in range(2):      # second pass: page cache warm, block pool filled
            rf = _capi.ReadFiles(f1, f2, n_threads=threads)
            t0 = time.perf_counter(); tot = 0
            while True:
                k = rf.next_batch(batch, L, out=bufs)[0]
                if k == 0:
                    break
                tot += k
            dt = time.perf_counter() - t0
            rf.close()
            best = max(best, tot / dt / 1e6)
        out["parser_only_mreads_s"] = best
        alpha, sm = _capi.quant_files_native(idx, f1, f2, batch=batch, max_read_len=L, threads=threads)
        alpha, sm = _capi.quant_files_native(idx, f1, f2, batch=batch, max_read_len=L, threads=threads)
        stream_s = max(sm["map_seconds"] - sm.get("map_setup_ms", 0.0) * 1e-3, 1e-9)
        out.update({"files_to_classes_mreads_s": sm["n_observed"] / sm["map_seconds"] / 1e6, "map_seconds": sm["map_seconds"],
                    "map_setup_ms": sm.get("map_setup_ms"), "files_to_classes_streaming_mreads_s": sm["n_observed"] / stream_s / 1e6,
                    "map_device_ms": sm["map_device_ms"], "em_seconds": sm["em_seconds"], "em_iters": sm["em_iters"],
                    "n_mapped": int(sm["n_mapped"]), "api": "sb_quant_files (C ABI): reader thread + GPU thread, then sb_em_optimize"})
        try:    # the same reads as .fastq.gz (what real data looks like): parallel inflate (csrc/pgzip.h)
            out["gz"] = stage_a_from_gz(idx, d, f1, f2, n, L, batch, threads)
        except Exception as e:  # noqa: BLE001
            out["gz"] = {"error": repr(e)}
        return out
    except Exception as e:  # noqa: BLE001  (an extra measurement must not lose the bench line)
        return {"error": repr(e)}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def stage_a_cpu(idx, p, left, right, budget_s, ncores):
    """CPU port (the product's serial forms compiled for the host, OpenMP over reads) on a bounded sample."""
    import hostmap_lib
    hostmap_lib.SO = os.path.join(scratch_dir(), "libhostmap.so")
    probe = min(20_000, left.shape[0])
    dt, _, _ = hostmap_lib.map_throughput(idx, p, left[:probe], right[:probe], 0, ncores)
    n = int(min(left.shape[0], max(probe, probe * budget_s / max(dt, 1e-3))))
    dt, na, c = hostmap_lib.map_throughput(idx, p, left[:n], right[:n], 0, ncores)
    return n / dt / 1e6, n, c


def bench_stage_a(args, rank, world, local, dist, W, peak, peak_src, ncores):
    import torch
    from salmon_b200 import _capi
    from salmon_b200._capi import Index, MapContext, map_default_params
    t0 = time.perf_counter()
    txps, flat, left, right = stage_a_workload(rank, small=args.sa_small)
    n, L = left.shape
    idx = Index(txps)
    info = idx.info()
    t_setup = time.perf_counter() - t0
    p = map_default_params()
    batch = min(SA["batch"], n)
    ctx = MapContext(idx, p, device=local, batch_cap=batch, max_read_len=L)
    _capi.pin(left); _capi.pin(right)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step(dev_ptrs=None):
        """one pass over this rank's n read pairs: all batches + finish()."""
        ctx.reset()
        dev_ms, seed_ms, seed_n, launches, ctr = 0.0, 0.0, 0, 0, None
        t0 = time.perf_counter()
        for s in range(0, n, batch):
            m = min(batch, n - s)
            if dev_ptrs is None:
                st = ctx.map_batch(left[s:s + m], right[s:s + m])
            else:
                st = ctx.map_batch_ptr(dev_ptrs[0] + s * L, dev_ptrs[1] + s * L, m, L)
            dev_ms += st.device_ms; seed_ms += st.seed_kernel_ms; seed_n += st.seed_kernel_launches
            launches = st.gpu_launches
        res = ctx.finish()
        wall = time.perf_counter() - t0
        return wall, dev_ms, seed_ms, seed_n, launches, res

    # ---- e2e: host (pinned) buffers through the C ABI, H2D inside, finish() (D2H of the class table) inside
    for _ in range(W):
        barrier(); step()
    e2e_s, launches0 = [], 0
    for _ in range(args.steps):
        barrier()
        wall, dev_ms, seed_ms, seed_n, launches, res = step()
        e2e_s.append(wall)
    # ---- inputs resident in HBM
    torch.cuda.set_device(local)
    dl = torch.from_numpy(left).cuda(); dr = torch.from_numpy(right).cuda()
    ctx.set_option("input_on_device", 1)
    sampler = ClockSampler(local); sampler.start(); sampler.wait_first()
    barrier(); launches = step((dl.data_ptr(), dr.data_ptr()))[4]
    sampler.mark()
    res_s, seed_ms_l, seed_n_l, dev_ms_l = [], [], 0, []
    launches_before = launches          # the library's counter is cumulative per context
    for _ in range(args.steps):
        barrier()
        wall, dev_ms, seed_ms, seed_n, launches, res = step((dl.data_ptr(), dr.data_ptr()))
        res_s.append(wall); seed_ms_l.append(seed_ms); seed_n_l = seed_n; dev_ms_l.append(dev_ms)
    launches_timed = launches - launches_before
    barrier()
    clocks_a = sampler.stop()
    c = res["counters"]

    def reduce_max(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64).cuda()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    res_t = reduce_max(statistics.mean(res_s)); e2e_t = reduce_max(statistics.mean(e2e_s))
    if rank != 0:
        ctx.close()
        return None, None
    d2h = sum(res[k].nbytes for k in ("off", "tids", "weights", "counts", "projected_counts", "eff_len", "unique_counts",
                                     "total_counts")) + (res["bins"].nbytes if res["bins"] is not None else 0)
    seed_launch_ms = statistics.mean(seed_ms_l) / max(seed_n_l, 1)
    frags_per_launch = n / max(seed_n_l, 1)
    seed_bytes = (n * 2 * L / 4 + c["lookups"] * 96 + c["postings"] * 8) / max(seed_n_l, 1)
    seed_achieved = seed_bytes / (seed_launch_ms / 1e3) / 1e9
    out = {
        "metric": "Mreads/s selective-align", "value": world * n / res_t / 1e6, "unit": "Mreads/s",
        "ms_per_step": res_t * 1e3, "higher_is_better": True, "scaling": "weak", "dtype": "u8/i32 (mapping), f64 (weights)",
        "steps_ms_rank0": {"resident": [round(x * 1e3, 2) for x in res_s], "e2e": [round(x * 1e3, 2) for x in e2e_s],
                           "resident_device_events": [round(x, 2) for x in dev_ms_l]},
        "timing": "value / e2e: host clock around the synchronous C-ABI calls of a step (sb_map_batch x batches + sb_map_finish), "
                  "barrier + synchronize on both sides, max over ranks -- it contains the device time (CUDA events on the "
                  "library's streams, resident_device_events, batches only) plus finish() and the host side of the calls, so it "
                  "cannot overstate the rate",
        "config": {"workload": f"configs[2] shape: synth_txome(seed=44, n_genes={SA['n_genes'] // (20 if args.sa_small else 1)}) = "
                               f"{len(txps)} transcripts / {flat[1].shape[0] / 1e6:.0f} Mb / {info['n_kmers'] / 1e6:.0f} M distinct 31-mers; "
                               f"{n} synthetic 2x{L} bp IU pairs per GPU per step (0.5% substitutions, 3% unmappable), "
                               f"batches of {batch}; a step = all batches + finish()",
                   "index_bytes": info["bytes"], "setup_s": t_setup,
                   "affinity_cores": len(_AFFINITY or []), "omp_num_threads": os.environ.get("OMP_NUM_THREADS"),
                   "l2": "index (7.9 GB) and per-step reads (419 MB) exceed L2",
                   "counters_per_step": c, "classes": int(len(res["counts"]))},
        "e2e": {"value": world * n / e2e_t / 1e6, "unit": "Mreads/s", "h2d_bytes_per_step": int(2 * n * L),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_t * 1e3,
                "api": "sb_map_batch x batches + sb_map_finish (C ABI, pinned host buffers)"},
        "gpu_launches": int(launches_timed), "gpu_launches_per_step": launches_timed / max(args.steps, 1),
        "clocks": clocks_a,
        "roofline": {"bound": "hbm", "kernel": "k_seed_chain_w", "achieved": seed_achieved, "peak": peak, "unit": "GB/s",
                     "frac": seed_achieved / peak, "peak_source": peak_src, "avg_launch_ms": seed_launch_ms,
                     "fragments_per_launch": frags_per_launch,
                     "algorithmic_bytes_per_launch": seed_bytes,
                     "traffic": stage_a_traffic(frags_per_launch),
                     "whole_stage_algorithmic_gbs": stage_a_algorithmic_bytes(n, L, c) / res_t / 1e9,
                     "note": "the kernel is latency/issue-bound (dependent hash-probe -> posting loads, warp-level sort "
                             "and scans), not bandwidth-bound: see DESIGN.md"},
    }
    if world == 1:
        v, ns, cc = stage_a_cpu(idx, p, left, right, args.cpu_budget, ncores)
        out["cpu_baseline"] = {"value": v, "unit": "Mreads/s", "cores": ncores, "kind": "port",
                               "sample": f"{ns} read pairs of the same workload, same index, OpenMP over reads",
                               "note": "NOT a credible reference baseline: the product's serial forms compiled for the host over the "
                                       "product's hash index, an order of magnitude below salmon's per-core rate; reported for "
                                       "completeness, no speed-up is claimed from it (DESIGN.md section 6)"}
        ctx.close()
        ctx = None
        if not args.no_files:
            out["from_files"] = stage_a_from_files(idx, left, right, batch, ncores)
    if ctx is not None:
        ctx.close()
    return out, res


DUMP_BYTES = 64 << 20


def class_order(res):
    """the classes of an sb_map_finish result sorted by label (transcripts, then range-factorisation bins): the device
    emits them in hash-table order, which differs from run to run"""
    off = res["off"].astype(np.int64).tolist()
    tids = res["tids"].tolist()
    bins = res["bins"].tolist() if res["bins"] is not None else None
    labels = [tids[a:b] + (bins[a:b] if bins is not None else []) for a, b in zip(off[:-1], off[1:])]
    return np.array(sorted(range(len(labels)), key=labels.__getitem__), dtype=np.int64)


def collect_outputs(alpha, alpha_e2e, stage_a_res):
    """What the last timed step of each path handed to its caller, by name:
      em_alpha, em_alpha_e2e  the abundances from sb_em_run (class table resident) and from sb_em_optimize (host buffers)
      stage_a_<name>          the per-transcript EM inputs from sb_map_finish
      stage_a_class_<name>    its class table in label order: per class sizes and counts, per entry tids, weights, bins;
                              a seeded sample of the classes if all of them would take the output past DUMP_BYTES"""
    out = {"em_alpha": alpha, "em_alpha_e2e": alpha_e2e}
    if stage_a_res is None:
        return out
    r = stage_a_res
    for k in ("projected_counts", "eff_len", "unique_counts", "total_counts"):
        out["stage_a_" + k] = r[k]
    off = r["off"].astype(np.int64)
    sizes = np.diff(off)
    fields = ("tids", "weights") + (("bins",) if r["bins"] is not None else ())
    order = class_order(r)
    room = DUMP_BYTES // 8 - 1024 - sum(a.size for a in out.values())      # float64 values left (1024: the .npy headers)
    cost = 2 + len(fields) * sizes[order]
    if cost.sum() > room:
        perm = np.random.default_rng(0).permutation(len(order))
        order = order[np.sort(perm[:np.searchsorted(np.cumsum(cost[perm]), room, side="right")])]
    sz = sizes[order]
    entries = np.repeat(off[:-1][order] - np.concatenate(([0], np.cumsum(sz)[:-1])), sz) + np.arange(sz.sum())
    out["stage_a_class_sizes"] = sz
    out["stage_a_class_counts"] = r["counts"][order]
    for k in fields:
        out["stage_a_class_" + k] = r[k][entries]
    return out


def dump_outputs(d, arrays):
    """every array as d/<name>.npy in float64 (integers below 2**53 are exact in it)"""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--em", action="store_true", help="plain EM instead of VBEM (not the headline)")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--nccl", action="store_true", help="N>1: per-iteration ncclAllReduce instead of the fused kernel")
    ap.add_argument("--no-stage-a", action="store_true", help="skip the Stage A (mapping) measurement")
    ap.add_argument("--sa-small", action="store_true", help="Stage A on a 20x smaller transcriptome (dev)")
    ap.add_argument("--no-files", action="store_true", help="skip the FASTQ-files -> classes measurement (row f1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the B200 arm's outputs")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    vbem = 0 if args.em else 1
    W = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    from salmon_b200.synth import synth_eq
    ncores = os.cpu_count() or 1
    workload = (f"configs[1] EM/VBEM-only: synth_eq(seed=1) C={C2['C']} classes, M={C2['M']} transcripts, "
                f"{ITERS_PER_STEP} forced {'VBEM' if vbem else 'EM'} iterations per step")
    # `config` is byte-identical in both arms (the driver compares them); arm-specific facts go to `details`
    config = {"workload": workload, "iters_per_step": ITERS_PER_STEP, "per_gpu_classes": C2["C"], "transcripts": C2["M"],
              "total_count": C2["total_count"], "algorithm": "VBEM" if vbem else "EM", "n_ranks": world}

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        eq, proj, eff, uniq = synth_eq(seed=1, **C2)
        rates, sample_iters = [], 0
        budget = max(2.0, min(args.cpu_budget, 120.0 / max(1, args.steps + args.warmup)))
        for i in range(args.warmup + args.steps):
            r, n, used, _ = cpu_port_rate(eq, proj, eff, uniq, vbem, budget, ncores)
            if i >= args.warmup:
                rates.append(r); sample_iters = n
        val = statistics.median(rates)
        line = {
            "impl": "reference", "metric": "EM iters/s", "value": val, "unit": "iters/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * ITERS_PER_STEP / val, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "details": {"note": "reference cannot be built here (Boost/oneTBB/pufferfish absent); CPU arm = in-repo "
                                "restatement parallelised like the reference (parallel_for over classes + CAS f64 adds), "
                                "OpenMP for oneTBB", "affinity_cores": len(_AFFINITY or []),
                        "step_rates": [round(x, 1) for x in rates]},
            "cpu_baseline": {"value": val, "unit": "iters/s", "cores": used, "kind": "port", "host_cores": ncores,
                             "sample": f"median over steps; each step = median of {CPU_REPEATS} runs of {sample_iters} "
                                       f"iterations of the same workload; thread count probed once per box "
                                       f"(best of all/64/32/16/8/serial, cached in a temp file), threads pinned"},
            "e2e": {"value": val, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        if not args.no_stage_a:
            from salmon_b200._capi import Index, map_default_params
            txps, flat, left, right = stage_a_workload(0, small=args.sa_small)
            idx = Index(txps)
            v, ns, cc = stage_a_cpu(idx, map_default_params(), left, right, max(4.0, min(args.cpu_budget, 20.0)), ncores)
            line["stage_a"] = {"metric": "Mreads/s selective-align", "value": v, "unit": "Mreads/s", "impl": "reference",
                               "cpu_baseline": {"value": v, "unit": "Mreads/s", "cores": ncores, "kind": "port",
                                                "sample": f"{ns} read pairs, {len(txps)} transcripts, OpenMP over reads",
                                                "note": "NOT a credible reference baseline (see DESIGN.md section 6)"}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ B200 arm
    from salmon_b200 import EMContext, default_params, _capi
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", rank=rank, world_size=world)
    ctx = EMContext(local)
    # per-rank class table (weak scaling): the eq-classes of this rank's read shard
    eq, proj, eff, uniq = synth_eq(seed=1 + rank, **C2)
    if world > 1:
        import torch
        # end-of-mapping reductions (SURVEY 8e): per-transcript masses are global
        tp = torch.from_numpy(proj).cuda(); dist.all_reduce(tp); proj = tp.cpu().numpy()
        tu = torch.from_numpy(uniq.astype(np.int64)).cuda(); dist.all_reduce(tu); uniq = tu.cpu().numpy().astype(np.uint64)
        te = torch.from_numpy(eff).cuda(); dist.broadcast(te, 0); eff = te.cpu().numpy()
        if args.nccl:
            uid = [_capi.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            ctx.comm_init(rank, world, uid[0])
        else:
            ctx.peer_setup(dist, C2["M"])
    for a in (eq.off, eq.tids, eq.weights, eq.counts, proj, eff, uniq):
        _capi.pin(a)
    p = default_params(use_vbem=vbem, min_iter=ITERS_PER_STEP, max_iter=ITERS_PER_STEP)

    def barrier():
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    # ---- device-resident: sb_em_run only
    ctx.upload(eq, proj, eff, uniq)
    ctx.prepare(p)
    sampler = ClockSampler(local); sampler.start(); sampler.wait_first()
    for _ in range(W):
        ctx.flush_l2(); barrier(); ctx.run()
    sampler.mark()
    run_ms, loop_ms, launches, loop_launches = [], [], 0, 0
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.flush_l2()
        barrier()
        st = ctx.run()
        run_ms.append(st.run_ms); loop_ms.append(st.loop_kernel_ms)
        launches += st.gpu_launches; loop_launches += st.loop_kernel_launches
    barrier()
    wall_resident = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    alpha, alpha_sum, ok = ctx.download()
    assert ok and st.iters == ITERS_PER_STEP
    # every valid class hands out exactly its count (size-independent sanity inside the bench)
    tot_counts = float(eq.counts.sum())
    if world > 1:
        import torch
        tc = torch.tensor([tot_counts], dtype=torch.float64).cuda(); dist.all_reduce(tc); tot_counts = tc.item()
    assert abs(alpha_sum - tot_counts) / tot_counts < 1e-9, (alpha_sum, tot_counts)

    # ---- end to end: sb_em_optimize, host buffers in/out
    e2e_ms = []
    for i in range(2 + args.steps):
        ctx.flush_l2()
        barrier()
        t0 = time.perf_counter()
        a2, st2, ok2 = ctx.optimize(eq, p, proj, eff, uniq)
        dt = time.perf_counter() - t0
        if i >= 2:
            e2e_ms.append(dt * 1e3)
    h2d = eq.off.nbytes + eq.tids.nbytes + eq.weights.nbytes + eq.counts.nbytes + proj.nbytes + eff.nbytes + uniq.nbytes
    d2h = alpha.nbytes

    def reduce_max(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64).cuda()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    step_ms = reduce_max(statistics.mean(run_ms))          # device time (CUDA events), max over ranks
    e2e_step_ms = reduce_max(statistics.mean(e2e_ms))
    loop_step_ms = reduce_max(statistics.mean(loop_ms))
    value = world * ITERS_PER_STEP / (step_ms / 1e3)
    e2e_value = world * ITERS_PER_STEP / (e2e_step_ms / 1e3)

    # ---- strong scaling (what a user of configs[1] gets from N GPUs): ONE 500k-class table split over the ranks
    strong = None
    if world > 1:
        from salmon_b200.synth import shard_classes
        eq_all, proj_a, eff_a, uniq_a = synth_eq(seed=1, **C2)
        sh = shard_classes(eq_all, rank, world)
        ctx.upload(sh, proj_a, eff_a, uniq_a)
        ctx.prepare(p)
        s_ms = []
        for i in range(2 + min(args.steps, 5)):
            ctx.flush_l2(); barrier()
            r = ctx.run()
            if i >= 2:
                s_ms.append(r.run_ms)
        s_step = reduce_max(statistics.mean(s_ms))
        strong = {"iters_per_s": ITERS_PER_STEP / (s_step / 1e3), "ms_per_step": s_step,
                  "workload": f"the seed=1 table ({C2['C']} classes) round-robin split over {world} ranks"}

    peak, peak_src = measured_peak()
    ctx.close()
    stage_a, stage_a_res = None, None
    if not args.no_stage_a:
        stage_a, stage_a_res = bench_stage_a(args, rank, world, local, dist, W, peak, peak_src, ncores)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    b_iter = algorithmic_bytes_per_iter(eq, bool(vbem))
    fused = world == 1 or not args.nccl
    kern_iters_per_launch = ITERS_PER_STEP if fused else 1
    avg_launch_ms = loop_step_ms if fused else loop_step_ms / ITERS_PER_STEP
    achieved = b_iter * kern_iters_per_launch / (avg_launch_ms / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic_r2.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get("dram_bytes_per_launch")
    cpu_val, cpu_n, cpu_used, cpu_rates = (cpu_port_rate(eq, proj, eff, uniq, vbem, args.cpu_budget, ncores)
                                           if world == 1 else (None, 0, 0, []))
    line = {
        "metric": "EM iters/s", "value": value, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
        "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config,
        "details": {"per_gpu_nnz": eq.nnz, "affinity_cores": len(_AFFINITY or []),
                   "l2": "flushed (memset > 2x L2) before every timed step; inside a step the table is re-swept "
                         "1000x and stays L2-resident, as in production",
                   "parallelism": "1 GPU" if world == 1 else
                   f"classes sharded over {world} GPUs (own table per rank), alpha all-reduced per iteration "
                   f"({'ncclAllReduce' if args.nccl else 'inside the persistent kernel over NVLink peer memory'}); "
                   f"value = {world} x iterations/s",
                   "kernel": "persistent cooperative k_em_persistent (1 launch per step)" if world == 1 else
                   ("k_em_p1 + k_em_p2_partial + ncclAllReduce + k_em_update per iteration" if args.nccl else
                    "k_em_persistent_mgpu: 1 cooperative launch per step per rank; partial alpha' pushed to owner slices as "
                    "flagged 16-byte lines over NVLink peer memory, theta' pushed back, no exchange barrier"),
                   "wall_s_resident_loop": wall_resident, "strong_scaling": strong},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "iters/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_step_ms, "api": "sb_em_optimize (C ABI, pinned host buffers)"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_iteration": b_iter,
                     "kernel": "k_em_persistent" if world == 1 else
                     ("k_em_p1+k_em_p2_partial+k_em_update" if args.nccl else "k_em_persistent_mgpu"),
                     "avg_launch_ms": avg_launch_ms, "iterations_per_launch": kern_iters_per_launch,
                     "note": "data is L2-resident by design, so DRAM traffic is far below the algorithmic bytes"},
    }
    if cpu_val is not None:
        line["cpu_baseline"] = {"value": cpu_val, "unit": "iters/s", "cores": cpu_used, "kind": "port",
                                "host_cores": ncores,
                                "sample": f"median of {CPU_REPEATS} runs of {cpu_n} iterations of the same workload; thread "
                                          f"count probed once per box (cached in a temp file, shared with the "
                                          f"reference arm), threads pinned",
                                "runs": [round(x, 1) for x in cpu_rates]}
    if stage_a is not None:
        line["stage_a"] = stage_a
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, collect_outputs(alpha, a2, stage_a_res))
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
