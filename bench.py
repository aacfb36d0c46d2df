#!/usr/bin/env python
"""bench.py -- RS encode GB/s at (n,k)=(2^20,2^19), 4 KiB blocks (BASELINE.json metric), on N B200s.

Own arm (default): one process per GPU (torchrun for N>1).  A step = one full encode (RS.cpp:41-63) of N=2^19 data
blocks x 4096 B -> 2^19 parity blocks.  Throughput convention is the reference's: bytes = 2*N*SIZE*4 per encode (RS.cpp:38).
  N = 1: the array is resident in HBM, the step is fastecc_b200_rs_encode_dev (three pass kernels).
  N > 1: ONE encode sharded over the N GPUs (BASELINE config 4; "scaling": "strong"): blocks dealt cyclically, the
         four-step transposes (TransposeMatrix, ntt.cpp:322-341,415,433,445) fused into the pass kernels' stores over
         peer memory (fastecc_b200/sharded.py).  Independent stripes per GPU (no data-path collective, weak scaling) are
         reported as the secondary block "stripes" of the same line.
Before anything is timed the result is checked: the parity of the reference's own fill (data0[i] = i % P, RS.cpp:28-29)
must hash (main.cpp:203-212) to the golden value of the unmodified reference, and for N > 1 the gathered sharded result
must equal the single-GPU encode bit for bit.  A mismatch aborts the run: no line is printed.

`--impl reference`: times the UNMODIFIED reference CPU encoder (oracle/_ref, compiled from /root/reference by
oracle/Makefile: AVX2 + OpenMP build, all host threads) on the same config; rank 0 only.

One JSON line on stdout (rank 0).  See DESIGN.md section 7 for how every field is measured.
`--dump-outputs DIR` also writes a fixed sample of the parity blocks of the last timed step to DIR/parity.npy.
"""
import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
P = 0xFFF00001
METRIC = "rs_encode_GBps_n2^20_k2^19_4KiB_blocks"
# hash (main.cpp:203-212) of the parity of fill A (data0[i] = i % P), recorded from the unmodified reference: SURVEY.md 8c,
# tests/golden/survey_8c.json "encode_fillA"; key = (log2 N, words per block)
GOLDEN_PARITY_HASH_FILL_A = {(7, 1024): 421122310, (11, 1024): 2634925848, (16, 1024): 147925734, (19, 1024): 4272226309, (7, 513): 56723226}
DUMP_ROWS = 1024                # parity blocks --dump-outputs writes: 8 MiB at 4 KiB blocks
DUMP_MAX_BYTES = 64 << 20


def workload_name(args):
    """The same string in both arms (the driver compares it); where the data lives is config.residency."""
    return "rs_encode N=2^%d data blocks -> 2^%d parity, %d-byte blocks, GF(0xFFF00001)" % (args.log_n, args.log_n, args.block_bytes)


def bind_to_gpu_numa_node(local_rank):
    """Run this process (and therefore its pinned allocations: first touch) on the CPUs of the NUMA node the GPU hangs off.
    Returns a short description; never fails."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:                 # nvml prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return "numa node unknown"
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "numa node %d has no allowed cpu" % node
        os.sched_setaffinity(0, cpus)
        return "numa node %d (%d cpus)" % (node, len(cpus))
    except Exception as e:                              # noqa: BLE001 -- binding is an optimisation
        return "not bound (%s)" % type(e).__name__


def profiled_traffic():
    """DRAM bytes (read + write) per ntt_pass_kernel launch from the committed `ncu --set full` capture of this workload
    (profiles/*_passes_A_BC_D.csv, highest round / version in the name), averaged over the three passes of an encode; None if absent."""
    import csv
    import glob
    import re

    def version(path):                      # r<round>_ncu_v<kernel version>_passes_A_BC_D.csv: newest round, then newest version
        m = re.search(r"r(\d+)_ncu_v(\d+)_passes", os.path.basename(path))
        return (int(m.group(1)), int(m.group(2))) if m else (-1, -1)
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_v*_passes_A_BC_D.csv")), key=version)
    if not files:
        return None, None
    try:
        rows = list(csv.reader(open(files[-1])))
        h, units, data = rows[0], rows[1], rows[2:]
        ir, iw = h.index("dram__bytes_read.sum"), h.index("dram__bytes_write.sum")
        scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        tot = [float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]] for r in data]
        return sum(tot) / len(tot), os.path.basename(files[-1])
    except Exception:
        return None, None


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=19, help="log2 of the number of data blocks (headline: 19)")
    ap.add_argument("--block-bytes", type=int, default=4096)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--mode", default="sharded", choices=["sharded", "sharded-a2a", "stripes"],
                    help="multi-GPU headline: ONE transform sharded over the GPUs with the exchange fused into the kernels' stores (default; strong scaling, "
                         "BASELINE config 4), the same with two NCCL all-to-alls, or only independent stripes (weak scaling)")
    ap.add_argument("--no-stripes", action="store_true", help="skip the secondary independent-stripes measurement of a multi-GPU run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the parity the last timed step computed to DIR/parity.npy (float64, a fixed "
                                                          "sample of at most %d blocks; see dump_rows) so two builds can be compared output for output" % DUMP_ROWS)
    return ap.parse_args()


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = sorted(s for s, p in zip(sm, pw) if p >= 0.6 * max(pw)) or sorted(sm)
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------- reference CPU arm
def load_ref_lib():
    path = os.path.join(ROOT, "oracle", "_ref", "libfastecc_ref.so")
    if not os.path.exists(path):
        return None
    r = ctypes.CDLL(path)
    r.ref_rs_encode.restype = None                      # RS.cpp:41-63 on a caller-supplied T** table
    r.ref_rs_encode.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t]
    r.ref_num_threads.restype = ctypes.c_int
    r.ref_build_flavour.restype = ctypes.c_char_p
    if hasattr(r, "ref_set_num_threads"):
        r.ref_set_num_threads.argtypes = [ctypes.c_int]; r.ref_set_num_threads.restype = None
    return r


def host_thread_candidates():
    """Thread counts worth trying for the CPU reference: one per physical core and one per hardware thread of this
    process's affinity mask (the reference blocks for the caches of a core: SMT siblings can hurt it, 1.8 s vs 4.6 s
    per encode on a 64-core / 128-thread host)."""
    cpus = sorted(os.sched_getaffinity(0))
    cores = set()
    for c in cpus:
        try:
            cores.add(open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c).read().strip())
        except OSError:
            cores.add(str(c))
    return sorted({max(1, len(cores)), len(cpus)})


def load_oracle_port():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    return oracle_lib.load_oracle()


def fill_index_mod_p(arr, chunk=1 << 24):
    """arr.flat[i] = i % P (the reference's fill, RS.cpp:28-29), in slices: no array-sized temporaries (eight ranks fill
    2 GiB each at the same time in the multi-GPU runs)."""
    import numpy as np
    flat = arr.reshape(-1)
    for lo in range(0, flat.size, chunk):
        hi = min(lo + chunk, flat.size)
        flat[lo:hi] = (np.arange(lo, hi, dtype=np.uint64) % P).astype(np.uint32)


def cpu_encode_runner(log_n, size_words, calibrate=True):
    """Returns (fn, kind, cores, label): fn() runs one full CPU encode of 2^log_n x size_words in place."""
    import numpy as np
    N = 1 << log_n
    buf = np.empty(N * size_words, dtype=np.uint32)
    fill_index_mod_p(buf)
    r = load_ref_lib()
    if r is not None:
        # T** data, RS.cpp:31-33; left permuted between steps like the reference leaves it
        tab = buf.ctypes.data + np.arange(N, dtype=np.uint64) * np.uint64(size_words * 4)
        fn = lambda _keep=buf: r.ref_rs_encode(tab.ctypes.data, N, size_words)      # noqa: E731
        note = ""
        cands = host_thread_candidates()
        if hasattr(r, "ref_set_num_threads") and calibrate:
            best = None
            for n in cands:                                   # give the reference its best thread count on this host
                r.ref_set_num_threads(n)
                if best is None:
                    fn()                                      # first touch / page faults are not part of the comparison
                t0 = time.perf_counter(); fn(); dt = time.perf_counter() - t0
                if best is None or dt < best[1]:
                    best = (n, dt)
            r.ref_set_num_threads(best[0])
            note = "; thread count picked from %s by one timed encode each" % cands
        return fn, "reference", int(r.ref_num_threads()), \
            "unmodified FastECC templates, %s+OpenMP build (oracle/_ref)%s" % (r.ref_build_flavour().decode(), note)
    o = load_oracle_port()
    return (lambda: o.oracle_rs_encode(buf.ctypes.data, N, size_words)), "port", int(o.oracle_num_threads()), "oracle/gfp_oracle.c (plain C port, OpenMP)"


def run_reference_arm(args):
    if args.dump_outputs:
        raise SystemExit("--dump-outputs writes the B200 arm's parity; the reference arm does not support it")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    os.environ.setdefault("OMP_WAIT_POLICY", "active")
    os.environ["OMP_NUM_THREADS"] = str(host_thread_candidates()[0])       # torchrun pins it to 1; cpu_encode_runner() then picks the better of cores / hardware threads
    size_words = args.block_bytes // 4
    N = 1 << args.log_n
    fn, kind, cores, label = cpu_encode_runner(args.log_n, size_words)
    for _ in range(max(1, min(args.warmup, 3))):
        fn()
    times = []
    budget_t0 = time.perf_counter()
    for _ in range(args.steps):
        t0 = time.perf_counter(); fn(); times.append(time.perf_counter() - t0)
        if time.perf_counter() - budget_t0 > 240:          # keep the whole run within a few minutes
            break
    total = sum(times)
    nbytes = 2.0 * N * size_words * 4
    value = nbytes * len(times) / total / 1e9
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "best_ms": 1e3 * min(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": workload_name(args), "residency": "host memory", "bytes_per_step": nbytes, "convention": "2*N*SIZE*4 bytes per encode (RS.cpp:38)"},
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": kind, "sample": "%d full encodes of the workload; %s" % (len(times), label)},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)
    return 0


def quick_cpu_baseline(args):
    """Bounded CPU sample for the own arm's cpu_baseline block: a few full encodes (about 10-30 s of CPU work at most)."""
    try:
        os.environ.setdefault("OMP_WAIT_POLICY", "active")
        os.environ["OMP_NUM_THREADS"] = str(host_thread_candidates()[0])
        size_words = args.block_bytes // 4
        fn, kind, cores, label = cpu_encode_runner(args.log_n, size_words)
        fn()
        times = []
        t_start = time.perf_counter()
        while len(times) < 5 and time.perf_counter() - t_start < 20:
            t0 = time.perf_counter(); fn(); times.append(time.perf_counter() - t0)
        nbytes = 2.0 * (1 << args.log_n) * size_words * 4
        return {"value": nbytes / min(times) / 1e9, "unit": "GB/s", "cores": cores, "kind": kind,
                "sample": "best of %d full encodes of the same workload (mean %.1f ms); %s" % (len(times), 1e3 * sum(times) / len(times), label)}
    except Exception as e:       # never let the baseline leg break the GPU measurement
        return {"value": None, "unit": "GB/s", "cores": 0, "kind": "unavailable", "sample": repr(e)}


# ---------------------------------------------------------------------------------------------------- B200 arm
def fill_a_rows(torch, dev, first_row, row_step, rows, S):
    """Rows first_row + l*row_step (l < rows) of the reference's fill data0[i] = i % P (RS.cpp:28-29) as an int32 CUDA tensor."""
    out = torch.empty((rows, S), dtype=torch.int32, device=dev)
    cols = torch.arange(S, device=dev, dtype=torch.int64)
    step = max(1, (1 << 24) // S)
    for lo in range(0, rows, step):
        hi = min(lo + step, rows)
        r = (torch.arange(lo, hi, device=dev, dtype=torch.int64) * row_step + first_row) * S
        out[lo:hi] = ((r[:, None] + cols[None, :]) % P).to(torch.int32)
    return out


def parity_hash(fe, t):
    """main.cpp:203-212 over the blocks of a device tensor, through the library's fastecc_b200_hash_u32."""
    import numpy as np
    return fe.reference_hash(t.cpu().numpy().view(np.uint32))


def check_golden(args, h, what):
    key = (args.log_n, args.block_bytes // 4)
    want = GOLDEN_PARITY_HASH_FILL_A.get(key) if args.block_bytes % 4 == 0 else None
    if want is not None and h != want:
        raise SystemExit("PARITY FAILURE (%s): hash %d != golden %d of the unmodified reference for N=2^%d, %d-byte blocks" % (what, h, want, key[0], args.block_bytes))
    return {"hash": h, "golden": want, "golden_match": None if want is None else True}


def dump_rows(N, S):
    """Global parity blocks written by --dump-outputs: every block when they fit, otherwise a sorted sample drawn with a fixed
    seed, so that runs with the same --log-n and --block-bytes write the same blocks."""
    import numpy as np
    rows = min(N, DUMP_ROWS, max(1, DUMP_MAX_BYTES // (8 * S)))
    if rows == N:
        return np.arange(N)
    return np.sort(np.random.default_rng(0).choice(N, rows, replace=False))


def write_dump(out_dir, sample):
    """sample: int32 CUDA tensor [rows, S] of parity words -> out_dir/parity.npy as float64 (exact: every word is < P < 2^53)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "parity.npy"), sample.cpu().numpy().view(np.uint32).astype(np.float64))


def per_kernel_roofline(fe, data, nbytes, peak, reps):
    """Per pass kernel: average duration over `reps` encodes with CUDA events between the launches (a separate loop right after
    the timed region: fastecc_b200_rs_encode_dev_timed synchronises the stream), algorithmic bytes = one read + one write of the array."""
    acc = None
    for _ in range(reps):
        t = fe.rs_encode_dev_timed(data)
        acc = [[n, ms] for n, ms in t] if acc is None else [[a[0], a[1] + ms] for a, (_, ms) in zip(acc, t)]
    acc = acc or []
    labels = {1: ["fused"], 2: ["A'", "B'"], 3: ["A", "BC", "D"]}.get(len(acc), [str(i) for i in range(len(acc))])
    out = []
    for lab, (name, ms) in zip(labels, acc):
        ms /= reps
        ach = nbytes / (ms * 1e-3) / 1e9
        out.append({"pass": lab, "kernel": name, "ms": round(ms, 4), "achieved": round(ach, 1), "frac": round(ach / peak, 4)})
    return out


def run_b200_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    numa = bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep NCCL's banner off stdout: rank 0 prints exactly one JSON line there
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import fastecc_b200 as fe
    fe.init(local)                      # raises if the CUDA library or an sm_100 GPU is missing: no fallback

    N, S = 1 << args.log_n, args.block_bytes // 4
    dev = torch.device("cuda", local)
    if args.mode in ("sharded", "sharded-a2a") and world > 1:
        return run_sharded(args, fe, rank, world, local, dev, numa)
    return run_single_or_stripes(args, fe, rank, world, local, dev, numa)


def time_stripes(args, fe, dev, world, data):
    """K encodes of this rank's own HBM-resident stripe between CUDA events; max over ranks.  Returns (ms, launches)."""
    import torch
    import torch.distributed as dist
    from fastecc_b200 import multirank

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(args.warmup, 3)):
        fe.rs_encode_dev(data)
    barrier()
    launches0 = fe.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        fe.rs_encode_dev(data)
    ev1.record()
    torch.cuda.synchronize()
    ms = multirank.max_over_ranks(ev0.elapsed_time(ev1), device=dev)          # a multi-GPU step takes as long as its slowest rank
    launches = fe.kernel_launches() - launches0
    barrier()
    return ms, launches


def run_single_or_stripes(args, fe, rank, world, local, dev, numa):
    import numpy as np
    import torch
    import torch.distributed as dist
    from fastecc_b200 import multirank
    N, S = 1 << args.log_n, args.block_bytes // 4
    nbytes = 2.0 * N * S * 4

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity first: the reference's own fill must give the reference's parity hash
    data = fill_a_rows(torch, dev, 0, 1, N, S)
    fe.rs_encode_dev(data)
    parity = {"device_resident": check_golden(args, parity_hash(fe, data), "device-resident encode")} if rank == 0 else None
    want_dev = data if not args.no_e2e else None                          # kept to compare the end-to-end result with
    data = fill_a_rows(torch, dev, 0, 1, N, S)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    ms, launches = time_stripes(args, fe, dev, world, data)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:             # data holds the parity of the last timed encode until the roofline loop below
        write_dump(args.dump_outputs, data[torch.from_numpy(dump_rows(N, S)).to(dev)])

    peak, peak_src = measured_peak()
    kernels = per_kernel_roofline(fe, data, nbytes, peak, max(3, min(args.steps, 10))) if rank == 0 else None
    del data

    # ---- end-to-end through the reference-facing host call (T** table, pinned host memory, H2D + D2H inside)
    e2e = None
    if not args.no_e2e:
        hptr = fe.lib().fastecc_b200_host_alloc(N * S * 4)
        if not hptr:
            raise SystemExit("pinned allocation failed")
        harr = np.ctypeslib.as_array((ctypes.c_uint32 * (N * S)).from_address(hptr)).reshape(N, S)
        fill_index_mod_p(harr)
        fe.EncodeReedSolomon_body(harr, N, S)                           # warm-up (allocates the device staging buffer) ...
        same = bool(torch.equal(torch.from_numpy(harr.view(np.int32)), want_dev.cpu()))       # ... and the parity check of this path
        if not same:
            raise SystemExit("PARITY FAILURE: fastecc_b200_rs_encode (host T** path) differs from the device-resident encode")
        if rank == 0:
            parity["host_api"] = dict(check_golden(args, fe.reference_hash(harr), "host T** encode"), equals_device_resident=True)
        del want_dev
        torch.cuda.empty_cache()
        fill_index_mod_p(harr)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            fe.EncodeReedSolomon_body(harr, N, S)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_s = multirank.max_over_ranks(e2e_s, device=dev)
        e2e = {"value": world * nbytes * args.e2e_steps / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": N * S * 4, "d2h_bytes_per_step": N * S * 4,
               "ms_per_step": 1e3 * e2e_s / args.e2e_steps, "api": "fastecc_b200_rs_encode(T** data, N, SIZE) on pinned host blocks", "host_numa": numa}
        del harr
        fe.lib().fastecc_b200_host_free(hptr)

    if rank == 0:
        traffic, traffic_src = profiled_traffic() if (args.log_n == 19 and args.block_bytes == 4096) else (None, None)
        top = max(kernels, key=lambda k: k["ms"]) if kernels else {"kernel": "small_dft_kernel", "pass": "single", "achieved": nbytes / (ms / args.steps * 1e-3) / 1e9,
                                                                   "frac": nbytes / (ms / args.steps * 1e-3) / 1e9 / peak}
        out = {
            "metric": METRIC, "value": world * nbytes * args.steps / (ms * 1e-3) / 1e9, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(args), "residency": "HBM (value) / pinned host memory (e2e)",
                       "bytes_per_step": nbytes, "convention": "2*N*SIZE*4 bytes per encode (RS.cpp:38)", "per_gpu_buffer_bytes": N * S * 4,
                       "l2": "inputs (2 GiB per GPU) are larger than L2; no flush needed", "parallelism": "independent stripe per GPU" if world > 1 else "single GPU",
                       "passes_per_encode": launches / max(args.steps, 1)},
            "roofline": {"bound": "hbm", "kernel": top["kernel"], "pass": top["pass"], "achieved": top["achieved"], "peak": peak, "unit": "GB/s", "frac": top["frac"],
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "per_kernel": kernels,
                         "encode_frac_of_compulsory_bytes": round(nbytes / (ms / args.steps * 1e-3) / 1e9 / peak, 4),
                         "note": "dominant (longest) pass kernel; algorithmic bytes per launch = 2*N*SIZE*4 (one read + one write of the array per pass); "
                                 "durations = CUDA events between the launches, averaged over a loop of encodes right after the timed region"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "parity": parity,
        }
        if e2e:
            out["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = quick_cpu_baseline(args)
        emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_sharded(args, fe, rank, world, local, dev, numa):
    """ONE encode of 2^log_n blocks sharded over the ranks (fastecc_b200/sharded.py): parity check, device-resident timing,
    per-phase times, end to end from pinned host shards, and the independent-stripes figure as a secondary block."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from fastecc_b200 import multirank, sharded
    N, S = 1 << args.log_n, args.block_bytes // 4
    rows = N // world
    nbytes = 2.0 * N * S * 4
    fused = args.mode == "sharded" and sharded.p2p_supported(N, world)
    enc, barrier_kind = None, None
    if fused:                                   # exchange fused into the kernels' stores over peer memory
        barrier_kind = os.environ.get("FASTECC_B200_SHARD_BARRIER", "flags")
        enc = sharded.P2PShardedEncoder(N, S, barrier=barrier_kind)
    else:                                       # local passes + two NCCL all-to-alls
        run_pass = sharded.gpu_pass_runner(N, world, rank)

    def step(t):
        if enc is None:
            return sharded.rs_encode_sharded(t, N, world, run_pass)
        if t is not enc.x:
            enc.x.copy_(t)
        return enc.encode()

    def sync():
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()

    # ---- parity first.  Global block l*G + rank is local row l; fill A = data0[i] = i % P over the GLOBAL array (RS.cpp:28-29).
    single = None
    if rank == 0:
        single = fill_a_rows(torch, dev, 0, 1, N, S)
        fe.rs_encode_dev(single)                                        # the single-GPU encode of the same array
    parity, note = None, None
    while True:
        mine = step(fill_a_rows(torch, dev, rank, world, rows, S)).clone()
        gathered = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
        dist.gather(mine, gathered, dst=0)
        verdict = torch.zeros(1, dtype=torch.int32, device=dev)
        if rank == 0:
            par = torch.empty((N, S), dtype=torch.int32, device=dev)
            for r in range(world):
                par[r::world] = gathered[r]
            gathered = None
            verdict[0] = 1 if bool(torch.equal(par, single)) else 0
        dist.broadcast(verdict, src=0)
        if int(verdict.item()) == 1:
            break
        if enc is not None and enc.barrier_kind == "flags":            # safety net: the kernel barrier is newer than the NCCL one
            note = "flag barrier gave a parity mismatch on this box; fell back to the NCCL all-reduce barrier"
            try:
                enc.close()
            except RuntimeError:                                        # a barrier timed out: that is why we are here
                pass
            enc = sharded.P2PShardedEncoder(N, S, barrier="nccl")
            barrier_kind = "nccl"
            continue
        raise SystemExit("PARITY FAILURE: the sharded encode over %d GPUs differs from the single-GPU encode" % world)
    if rank == 0:
        parity = {"sharded": dict(check_golden(args, parity_hash(fe, par), "sharded encode"), equals_single_gpu_encode=True)}
        if note:
            parity["note"] = note
        del par, single
        torch.cuda.empty_cache()
    sync()

    x = fill_a_rows(torch, dev, rank, world, rows, S)
    for _ in range(max(args.warmup, 3)):
        x = step(x)
    sync()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start(); time.sleep(0.25)
    launches0 = fe.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    ev0.record()
    for _ in range(args.steps):
        x = step(x)
    ev1.record()
    torch.cuda.synchronize()
    ms = multirank.max_over_ranks(ev0.elapsed_time(ev1), device=dev)
    launches = fe.kernel_launches() - launches0
    clocks = sampler.stop() if sampler else None
    sync()
    if fused:
        enc.check()                             # no barrier timed out: the ranks stayed in step
    if args.dump_outputs:                       # x: this rank's rows of the last timed encode (global block l*G + rank = row l)
        g = torch.from_numpy(dump_rows(N, S)).to(dev)
        owned = g % world == rank
        sample = torch.zeros((g.numel(), S), dtype=torch.int32, device=dev)
        sample[owned] = x[g[owned] // world]
        dist.reduce(sample, dst=0)              # one rank contributes each row, the others zeros
        if rank == 0:
            write_dump(args.dump_outputs, sample)
    phases = None
    if fused:                                   # more encodes with events between the phases (max over ranks of the mean per phase)
        names = ["pass_A", "barrier_1", "pass_BC", "barrier_2", "pass_D"]
        acc = [0.0] * 5
        reps = 5
        for _ in range(reps):
            evs = []
            enc.encode(events=evs)
            torch.cuda.synchronize()
            for i in range(5):
                acc[i] += evs[i].elapsed_time(evs[i + 1]) / reps
            sync()
        phases = {n: round(multirank.max_over_ranks(v, device=dev), 4) for n, v in zip(names, acc)}

    # ---- end to end: every rank holds its shard in pinned host memory (allocated on its GPU's NUMA node)
    e2e = None
    if fused and not args.no_e2e:
        hptr = fe.lib().fastecc_b200_host_alloc(rows * S * 4)
        if not hptr:
            raise SystemExit("pinned allocation failed")
        harr = np.ctypeslib.as_array((ctypes.c_uint32 * (rows * S)).from_address(hptr)).reshape(rows, S)
        shard_cpu = fill_a_rows(torch, dev, rank, world, rows, S).cpu().numpy().view(np.uint32)
        harr[:] = shard_cpu
        enc.encode_host(harr)                                           # warm-up and parity check of this path
        ok = torch.tensor([1 if bool(torch.equal(torch.from_numpy(harr.view(np.int32)), mine.cpu())) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) != 1:
            raise SystemExit("PARITY FAILURE: sharded encode_host (pinned host shards) differs from the device-resident sharded encode")
        if rank == 0:
            parity["sharded_host_api"] = {"equals_device_resident_sharded": True}
        harr[:] = shard_cpu
        sync()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            enc.encode_host(harr)
        torch.cuda.synchronize()
        e2e_s = multirank.max_over_ranks(time.perf_counter() - t0, device=dev)
        e2e = {"value": nbytes * args.e2e_steps / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": N * S * 4, "d2h_bytes_per_step": N * S * 4,
               "ms_per_step": 1e3 * e2e_s / args.e2e_steps, "host_numa_rank0": numa,
               "api": "P2PShardedEncoder.encode_host: every rank's N/G blocks in pinned host memory, column-chunked H2D / 3 sharded passes / D2H pipeline; bytes are the totals over all ranks"}
        del harr, shard_cpu
        fe.lib().fastecc_b200_host_free(hptr)
        sync()
    del mine

    # ---- secondary: independent stripes (one full 2^log_n encode per GPU, no data-path collective)
    stripes = None
    if not args.no_stripes:
        data = fill_a_rows(torch, dev, 0, 1, N, S)
        sms, _ = time_stripes(args, fe, dev, world, data)
        del data
        stripes = {"value": world * nbytes * args.steps / (sms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": sms / args.steps, "scaling": "weak",
                   "what": "every GPU encodes its own independent 2^%d-block stripe (communication-free row of SURVEY 8e); aggregate over %d GPUs" % (args.log_n, world)}

    if rank == 0:
        a2a_bytes = 2.0 * (world - 1) / world * (N * S * 4 / world)           # sent per GPU per encode (two exchanges)
        link = 770.0                                                          # GB/s per direction per GPU, measured peer copy (B200_PROFILING.md)
        t_link = a2a_bytes / (link * 1e9)
        step_s = ms / args.steps * 1e-3
        out = {
            "metric": METRIC, "value": nbytes / step_s / 1e9, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(args), "residency": "HBM, N/G blocks per GPU (value) / pinned host shards (e2e)",
                       "bytes_per_step": nbytes, "convention": "2*N*SIZE*4 bytes per encode (RS.cpp:38)",
                       "parallelism": ("ONE transform over %d GPUs: cyclic blocks, 3 passes; passes A and BC store every output row into its owner's HBM over NVLink "
                                       "(peer-mapped, CUDA IPC), 2 barriers between the passes" % world
                                       if fused else "ONE transform over %d GPUs: cyclic blocks, 3 local passes + 2 NCCL all-to-all" % world),
                       "barrier": ({"flags": "one-warp kernel over the peer mappings (fastecc_b200_shard_barrier; no NCCL on the data path)",
                                    "nccl": "one-word NCCL all-reduce"}.get(barrier_kind) if fused else None),
                       "l2": "local arrays (%.0f MiB per GPU) exceed L2" % (N * S * 4 / world / 2**20)},
            "roofline": {"bound": "nvlink", "kernel": "ntt_pass_kernel<9,1,2> (A) + ntt_pass_kernel<10,2,2> (BC): the instantiations whose stores pick a destination GPU",
                         "achieved": a2a_bytes / step_s / 1e9, "peak": link, "unit": "GB/s",
                         "frac": t_link / step_s, "traffic": None,
                         "note": "bytes each GPU sends to its peers per encode (2 exchanges of (G-1)/G of the local array) / step time, against the measured 770 GB/s per-direction peer bandwidth"},
            "gpu_launches": int(launches), "clocks": clocks, "parity": parity,
        }
        if phases:
            out["phases_ms_max_over_ranks"] = phases
        if e2e:
            out["e2e"] = e2e
        if stripes:
            out["stripes"] = stripes
        emit(out)
    if fused:
        enc.close()
    dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def guard_stdout():
    """Libraries write banners to stdout (torch prints "NCCL version ..." when the first communicator is created).  The
    contract is ONE JSON line there, so file descriptor 1 points at stderr until emit() prints the result."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(obj), flush=True)
    if _REAL_STDOUT is not None:
        os.dup2(2, 1)


def main():
    args = parse_args()
    guard_stdout()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
