#!/usr/bin/env python
"""bench.py — headline benchmark: sites/s of popgenWindows (pi + Fst + Dxy) on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference command line on the host cores
    python bench.py ... --dump-outputs DIR                   # + the rows of the last timed step, to compare two builds

Workload (BASELINE.json configs[1], "C2"): 4 populations x 50 diploid samples (H = 400 haplotypes), 10 M synthetic sites per
GPU, -w 50000 coordinate windows (~5000 sites each), -m 100, minData 0.01.  A "step" is one pass of the hot path (site pass ->
window statistics -> rows on the host) over that batch.

  value           whole-job sites/s, matrix resident in HBM, NO missing genotypes: every window takes the closed-form
                  allele-count path (K1, the HBM-roofline kernel)
  value_missing   the same with 2 % missing genotypes — what real data looks like: every window is "ragged" and takes the
                  pairwise path (K2: tcgen05 int8 Gram kernels); roofline_missing describes its kernels
  e2e             value's workload through the public API from pinned HOST buffers (H2D + transcode + statistics + D2H)
  c3 / c4 / c5    the other BASELINE.json configs as first-class legs: C3 ABBABABAwindows strong scaling (10 M sites over the
                  N GPUs), C4 distMat 500 diploid samples x 2 M sites (N = 1), C5 freq.py + popgenWindows 8 x 100 samples,
                  12.5 M sites per GPU, --windType sites.  Every multi-GPU leg checks the gathered rows against a single-GPU
                  computation of the same shards inside the run ("rows_equal_single_gpu").
  cpu_baseline    the unmodified reference command line (oracle/_ref/popgenWindows.py, staged by oracle/build_ref.py) on a
                  bounded sample of the workload, best of -T in {1, 8, all cores}; falls back to the loop-faithful port
                  (oracle/ref_port.py) only if the staged scripts are missing

Multi-GPU: one process per GPU (torchrun); every rank owns its own shard, no data-path collective, the per-window records are
all-gathered once per step by the engine's native NCCL call.  Time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "sites/sec popgenWindows (pi+Fst+Dxy)"
N_POPS, SAMPLES_PER_POP, PLOIDY = 4, 50, 2
WIND_SIZE, MIN_SITES, MIN_DATA = 50000, 100, 0.01
SEED = 20260923 + 2
REF_DIR = os.path.join(REPO, "oracle", "_ref")


def env_int(name, dflt):
    try:
        return int(os.environ.get(name, dflt))
    except ValueError:
        return dflt


# ------------------------------------------------------------------------------------------------
# clocks sampled DURING the timed regions
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.samples.append((time.perf_counter(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()          # exactly the process we started
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, intervals):
        sm, mx, reasons = [], [], set()
        for t, line in self.samples:
            if not any(a <= t <= b for a, b in intervals):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# the workload as .geno text (for the reference command line and the from-text legs)
# ------------------------------------------------------------------------------------------------
def geno_text(spec, n_sites, pos_seed):
    """The synthetic matrix as the bytes of a phased .geno file (vectorised: ~1 s per 100 MB)."""
    from genomics_general_b200 import synth
    gt = synth.synth_genotypes(spec, 0, n_sites)
    pos = synth.synth_positions(n_sites, seed=pos_seed)
    nS = spec.n_samples
    txt = np.empty((n_sites, 5 + 9 + nS * 4 + 1), dtype=np.uint8)
    txt[:, :5] = np.frombuffer(b"chr1\t", dtype=np.uint8)
    txt[:, 5:14] = (pos[:, None].astype(np.int64) // 10 ** np.arange(8, -1, -1)[None, :]) % 10 + 48
    ch = np.frombuffer(b"ACGTN", dtype=np.uint8)[np.where(gt < 0, 4, gt)]
    body = txt[:, 14:14 + nS * 4].reshape(n_sites, nS, 4)
    body[:, :, 0] = 9                                                    # tab
    body[:, :, 1] = ch[:, 0::2]
    body[:, :, 2] = ord("|")
    body[:, :, 3] = ch[:, 1::2]
    txt[:, -1] = 10
    return ("#CHROM\tPOS\t" + "\t".join(spec.sample_names()) + "\n").encode() + txt.tobytes(), gt


def write_workload_files(tmpdir, n_sites, miss, seed):
    from genomics_general_b200 import synth
    spec = synth.SynthSpec(N_POPS, SAMPLES_PER_POP, PLOIDY, seed=seed, miss=miss)
    text, _ = geno_text(spec, n_sites, seed)
    gpath = os.path.join(tmpdir, "c2_%d_%g.geno" % (n_sites, miss))
    with open(gpath, "wb") as f:
        f.write(text)
    ppath = gpath + ".pops"
    with open(ppath, "wt") as f:
        for i, nm in enumerate(spec.sample_names()):
            f.write("%s pop%d\n" % (nm, i // SAMPLES_PER_POP))
    return gpath, ppath


# ------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference command line
# ------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def have_reference():
    return os.path.exists(os.path.join(REF_DIR, "popgenWindows.py")) and os.path.exists(os.path.join(REF_DIR, "genomics.py"))


def run_reference_cli(gpath, ppath, out, threads, timeout=1500):
    """python oracle/_ref/popgenWindows.py -w 50000 -m 100 -f phased -T t ...  -> wall seconds"""
    cmd = [sys.executable, os.path.join(REF_DIR, "popgenWindows.py"), "-w", str(WIND_SIZE), "-m", str(MIN_SITES), "-g", gpath,
           "-o", out, "-f", "phased", "-T", str(threads), "--popsFile", ppath]
    for k in range(N_POPS):
        cmd += ["-p", "pop%d" % k]
    t0 = time.perf_counter()
    r = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, timeout=timeout)
    dt = time.perf_counter() - t0
    if r.returncode != 0:
        raise RuntimeError("reference command line failed: %s" % r.stderr[-500:])
    return dt


def reference_sweep(tmpdir, miss, budget_s=30.0):
    """Bounded sample of the C2 workload through the reference CLI: -T in {1, 8, cores}; returns the cpu_baseline dict."""
    cores = host_cores()
    L = env_int("PG_BENCH_CPU_WINDOW_SITES", 5000)
    out = os.path.join(tmpdir, "ref_out.csv")
    g1, p1 = write_workload_files(tmpdir, 1 * L, miss, SEED + 31)
    t1 = run_reference_cli(g1, p1, out, 1)                          # -T 1 on ONE window (the rest scale linearly in windows)
    rates = {"1": L / t1}
    cand = sorted({t for t in (8, min(cores, 16), cores) if t > 1})
    # sample size: as many windows as the widest -T, bounded so that the sweep stays inside the budget at the -T 1 rate / 4
    nwin = max(2, min(max(cand), int(budget_s * (L / t1) * 4 / L) or 2, 16))
    gN, pN = write_workload_files(tmpdir, nwin * L, miss, SEED + 32)
    best_t, best_rate = 1, rates["1"]
    spent = t1
    for t in cand:
        if spent > 2.5 * budget_s:
            break
        dt = run_reference_cli(gN, pN, out, t)
        spent += dt
        rates[str(t)] = nwin * L / dt
        if rates[str(t)] > best_rate:
            best_t, best_rate = t, rates[str(t)]
    return {"value": best_rate, "unit": "sites/s", "cores": best_t, "kind": "reference",
            "sample": "unmodified reference popgenWindows.py (oracle/_ref, staged by oracle/build_ref.py) from .geno text: "
                      "-T 1 on 1 window, -T %s on %d windows of %d sites of the C2 shape, miss=%g; best = -T %d; "
                      "host has %d logical CPUs" % (",".join(str(c) for c in cand), nwin, L, miss, best_t, cores),
            "rates_by_T": rates, "host_cpus": cores, "miss": miss}, (gN, pN, nwin * L, best_t)


def port_sample(miss, windows, L):
    """fallback when oracle/_ref is absent: the loop-faithful port of the numeric core (no parsing)"""
    import warnings
    from genomics_general_b200 import synth
    from oracle import ref_port                                  # the checker, timed as the CPU baseline
    spec = synth.SynthSpec(N_POPS, SAMPLES_PER_POP, PLOIDY, seed=SEED, miss=miss)
    t = time.perf_counter()
    for k in range(windows):
        g = synth.synth_genotypes(spec, k * L, L)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref_port.popgen_window_port(g, spec.hap_pop(), N_POPS, MIN_SITES, MIN_DATA)
    dt = time.perf_counter() - t
    return {"value": windows * L / dt, "unit": "sites/s", "cores": 1, "kind": "port",
            "sample": "%d windows x %d sites, oracle/ref_port.py (numeric core only, one process), miss=%g" % (windows, L, miss),
            "miss": miss}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, all host threads it can use."""
    if rank != 0:
        return
    tmpdir = tempfile.mkdtemp(prefix="pg_ref_")
    cfg = workload_config(args, world)
    if have_reference():
        base, (gN, pN, n_sites, best_t) = reference_sweep(tmpdir, 0.0, budget_s=20.0)
        out = os.path.join(tmpdir, "ref_out.csv")
        for _ in range(max(args.warmup - 3, 0)):                  # the -T sweep above already ran the command line 3-4 times
            run_reference_cli(gN, pN, out, best_t)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            run_reference_cli(gN, pN, out, best_t)
        dt = time.perf_counter() - t0
        value = n_sites * args.steps / dt
        cpu = dict(base, value=value)
        cpu["sample"] += "; timed: %d runs of the -T %d command line on %d sites each" % (args.steps, best_t, n_sites)
    else:
        t0 = time.perf_counter()
        cpu = port_sample(0.0, max(args.steps, 1), 2000)
        dt = time.perf_counter() - t0
        value = cpu["value"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "sites/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": cfg, "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(args, world):
    """Pure function of the arguments: identical in both arms."""
    H = N_POPS * SAMPLES_PER_POP * PLOIDY
    return {"workload": "C2 popgenWindows: %d pops x %d diploid samples (H=%d), %d sites per GPU, -w %d coordinate "
                        "windows, -m %d, minData %g" % (N_POPS, SAMPLES_PER_POP, H, args.sites, WIND_SIZE, MIN_SITES, MIN_DATA),
            "sites_per_gpu": args.sites, "haplotypes": H,
            "sharding": "windows (one shard per GPU), one all-gather of rows" if world > 1 else "single GPU",
            "l2": "inputs (%.1f GB per GPU) are larger than L2; no flush needed" % (args.sites * H / 1e9)}


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def quiet_stdout():
    """Libraries (NCCL's version banner, torchrun notices) may write to fd 1; the contract is ONE JSON line on
    stdout.  Route fd 1 to stderr for the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def rows_equal(a: dict, b: dict, keys, rtol=0.0):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        if x.shape != y.shape:
            return False
        if rtol == 0.0:
            if not np.array_equal(x, y, equal_nan=True):
                return False
        elif not np.allclose(x, y, rtol=rtol, atol=1e-300, equal_nan=True):
            return False
    return True


DUMP_KEYS = ("sites", "pos_sum", "path", "pi", "dxy", "fst")
DUMP_LIMIT = 60_000_000          # bytes of array data: the files stay below 64 MB, .npy headers included


def dump_outputs(directory, legs, limit=DUMP_LIMIT):
    """Window rows of the last timed step of each leg as <directory>/<leg>_<key>.npy (float64; the integer columns are
    below 2**53).  Past `limit` bytes in all, every leg keeps a seeded sample of its windows, listed in <leg>_window.npy."""
    os.makedirs(directory, exist_ok=True)
    total = sum(np.asarray(rows[k]).size * 8 for rows in legs.values() for k in DUMP_KEYS)
    scale = limit / (total + 8 * sum(len(rows["sites"]) for rows in legs.values()))     # + the window index
    for leg, rows in legs.items():
        W = len(rows["sites"])
        keep = None
        if total > limit:
            n = max(1, int(W * scale))
            keep = np.sort(np.random.default_rng(SEED).choice(W, size=n, replace=False))
            np.save(os.path.join(directory, "%s_window.npy" % leg), keep.astype(np.float64))
        for k in DUMP_KEYS:
            a = np.asarray(rows[k], dtype=np.float64)
            np.save(os.path.join(directory, "%s_%s.npy" % (leg, k)), a if keep is None else a[keep])


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--sites", type=int, default=env_int("PG_BENCH_SITES", 10_000_000))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-legs", action="store_true", help="skip the C3 / C4 / C5 / text legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the window rows of the last timed step of the two C2 legs as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    from genomics_general_b200 import multigpu, synth, windows
    from genomics_general_b200.engine import Engine, PinnedArray

    dist = None
    dev = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local_rank)
        dev = torch.device("cuda", local_rank)
        dist.init_process_group(backend="nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_counts(n):
        if dist is None:
            return [int(n)]
        import torch
        cnt = torch.tensor([int(n)], dtype=torch.int64, device=dev)
        allc = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(allc, cnt)
        return [int(c.item()) for c in allc]

    S, P = args.sites, N_POPS
    H = N_POPS * SAMPLES_PER_POP * PLOIDY
    eng = Engine(local_rank)
    sampler = ClockSampler(local_rank)
    sampler.start()
    intervals = []
    if dist is not None:
        import torch
        # NCCL communicator of the engine itself: rank 0 creates the id, torch.distributed only carries it
        id_t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            id_t.copy_(torch.frombuffer(bytearray(eng.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(id_t, 0)
        eng.nccl_init(world, rank, bytes(id_t.cpu().numpy().tobytes()))

    def positions(n):
        pos = np.empty(n, dtype=np.int32)
        step = 1 << 22
        for s0 in range(0, n, step):
            m = min(step, n - s0)
            eng.download(s0, m, want_geno=False, into_pos=pos[s0:s0 + m])
        return pos

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        l0 = eng.launch_count()
        t0 = time.perf_counter()
        tms = []
        for _ in range(steps):
            fn()
            tms.append(eng.last_timings())
        dt_local = time.perf_counter() - t0          # every step ends with a device->host read (synchronised)
        barrier()
        intervals.append((t0, t0 + dt_local))
        return max_over_ranks(dt_local), tms, eng.launch_count() - l0

    def mean_ms(tms):
        keys = []
        for t in tms:
            for k in t:
                if k not in keys:
                    keys.append(k)
        return {k: float(np.mean([t[k]["ms"] for t in tms if k in t])) for k in keys}

    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        mp_ = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        peak, peak_src = float(mp_["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        pass

    # =============== C2, resident matrix ===============
    def c2_leg(miss, steps, warmup):
        spec = synth.SynthSpec(N_POPS, SAMPLES_PER_POP, PLOIDY, seed=SEED + 1000 * rank, miss=miss)
        eng.synth_fill(spec, S)
        eng.set_pops(spec.hap_pop(), P)
        pos = positions(S)
        lo, hi = windows.sliding_coord_windows(np.zeros(S, dtype=np.int32), ["chr1"], pos, WIND_SIZE).ranges()
        eng.set_windows(lo, hi)
        counts = all_counts(len(lo))
        w_max = max(max(counts), 1)
        table = PinnedArray((world * w_max, eng.popgen_record_width()), np.float64) if dist is not None else None

        def step():
            if dist is not None:
                # one C-ABI call: site pass -> finalize -> ncclAllGather (native, same stream, in place) -> D2H of the table
                eng.popgen_allgather(w_max, table.array, MIN_SITES, MIN_DATA)
                return table.array
            return eng.popgen(MIN_SITES, MIN_DATA)
        dt, tms, launches = timed(step, steps, warmup)
        # the same K steps PIPELINED: the exchange + read-back of batch k run on a side stream under the site pass of batch
        # k+1 (pg_popgen_gather_begin / _end, two slots) — every batch's table still reaches the host inside the timed region
        def pipelined():
            eng.popgen_gather_begin(w_max, 0, MIN_SITES, MIN_DATA)
            for k in range(1, steps):
                eng.popgen_gather_begin(w_max, k & 1, MIN_SITES, MIN_DATA)
                eng.popgen_gather_end(w_max, (k - 1) & 1)
            return eng.popgen_gather_end(w_max, (steps - 1) & 1)
        pipelined()
        barrier()
        l0 = eng.launch_count()
        t0 = time.perf_counter()
        last = pipelined()
        dtp_local = time.perf_counter() - t0
        barrier()
        intervals.append((t0, t0 + dtp_local))
        dt_pipe = max_over_ranks(dtp_local)
        launches_pipe = eng.launch_count() - l0
        last = np.array(last)                        # the slot is pinned memory that later batches overwrite
        ref_tab = step()
        if dist is not None:
            pipe_equal = bool(np.array_equal(last.view(np.uint64), np.asarray(ref_tab).view(np.uint64)))
            out_rows = multigpu.unpack_device_records(multigpu.gathered_rows(last, counts, w_max), P)
        else:
            out_rows = multigpu.unpack_device_records(last[:len(lo)], P)
            pipe_equal = rows_equal(ref_tab, out_rows, ("sites", "pos_sum", "path", "pi", "dxy", "fst"))
        # correctness of the gathered rows: rank 0 recomputes every rank's shard alone
        equal = None
        if dist is not None:
            gathered = multigpu.unpack_device_records(multigpu.gathered_rows(table.array.copy(), counts, w_max), P)
            if rank == 0:
                equal, off = True, 0
                for q in range(world):
                    sq = synth.SynthSpec(N_POPS, SAMPLES_PER_POP, PLOIDY, seed=SEED + 1000 * q, miss=miss)
                    eng.synth_fill(sq, S)
                    eng.set_pops(sq.hap_pop(), P)
                    lq, hq = windows.sliding_coord_windows(np.zeros(S, dtype=np.int32), ["chr1"], positions(S), WIND_SIZE).ranges()
                    eng.set_windows(lq, hq)
                    one = eng.popgen(MIN_SITES, MIN_DATA)
                    part = {k: gathered[k][off:off + counts[q]] for k in ("sites", "pos_sum", "path", "pi", "dxy", "fst")}
                    equal = equal and rows_equal(one, part, ("sites", "pos_sum", "path", "pi", "dxy", "fst"))
                    off += counts[q]
                eng.synth_fill(spec, S)
                eng.set_pops(spec.hap_pop(), P)
                eng.set_windows(lo, hi)
            barrier()
        paths = np.bincount(eng.popgen(MIN_SITES, MIN_DATA)["path"], minlength=3).tolist()
        return dict(dt=dt, tms=tms, launches=launches, steps=steps, W=len(lo), lo=lo, hi=hi, step=step, equal=equal,
                    paths=paths, table=table, dt_pipe=dt_pipe, launches_pipe=launches_pipe, pipe_equal=pipe_equal,
                    out_rows=out_rows)

    A = c2_leg(0.0, args.steps, args.warmup)
    value_sync = world * S * args.steps / A["dt"]
    value = world * S * args.steps / A["dt_pipe"]
    kernel_ms = mean_ms(A["tms"])
    k1_ms = kernel_ms.get("k1_popgen", float("nan"))

    # =============== e2e from pinned host buffers ===============
    e2e = None
    if not args.no_e2e:
        hg = PinnedArray((S, H), np.int8)
        hp = PinnedArray((S,), np.int32)
        slab = 1 << 20
        for s in range(0, S, slab):
            n = min(slab, S - s)
            eng.download(s, n, into_geno=hg.array[s:s + n], into_pos=hp.array[s:s + n])

        def step_e2e():
            eng.upload(hg.array, hp.array)            # H2D from pinned memory + device transcode
            eng.set_windows(A["lo"], A["hi"])
            return A["step"]()                        # statistics + D2H of the rows (+ all-gather when N > 1)

        e_steps = max(3, min(args.steps, 10))
        dt_e, _, _ = timed(step_e2e, e_steps, 1)
        npairs = P * (P - 1) // 2
        e2e = {"value": world * S * e_steps / dt_e, "unit": "sites/s", "h2d_bytes_per_step": int(S) * (H + 4),
               "d2h_bytes_per_step": int(A["W"]) * (8 * (P + 2 * npairs) + 20), "steps": e_steps,
               "ms_per_step": 1e3 * dt_e / e_steps}
        hg.close()
        hp.close()

    # =============== C2 with 2 % missing genotypes: the pairwise path ===============
    m_steps = max(3, min(args.steps, 10))
    B = c2_leg(0.02, m_steps, 2)
    value_missing = world * S * m_steps / B["dt_pipe"]
    value_missing_sync = world * S * m_steps / B["dt"]
    kernel_ms_missing = mean_ms(B["tms"])
    pair_macs = None
    roofline_missing = None
    try:
        km = kernel_ms_missing
        dom = max((k for k in km if k.startswith(("k2t_", "k2_"))), key=lambda k: km[k])
        # tensor work of the two Gram kernels: rows x columns of the upper-triangular 128-row tile groups x K bytes
        tiles = lambda R: sum(128 * (R - a) for a in range(0, R, 128))      # noqa: E731  accumulator cells computed
        n_var = None
        macs_n = tiles(208) * S                                            # 200 sample rows (padded to 208), K = every site
        gram_ms = km.get("k2t_gram_n", 0.0) + km.get("k2t_gram_diff", 0.0)
        sm_clock = 1.965e9
        int8_peak = 148 * 8192 * sm_clock                                   # measured: M128 N256 K32 per 128 cycles per SM
        vc = "k2t_valid_class"                                              # the chain's HBM-bound kernel
        roofline_missing = {
            "bound": "hbm", "kernel": vc, "kernel_ms": km[vc], "longest_kernel": dom,
            "achieved": S * (H + 4) / (km[vc] * 1e-3) / 1e9,
            "peak": peak, "unit": "GB/s",
            "frac": S * (H + 4) / (km[vc] * 1e-3) / 1e9 / peak,
            "traffic": None, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": S * (H + 4),
            "note": "the pairwise path is a chain of kernels, none above 0.9 ms: k2t_valid_class re-reads the resident matrix "
                    "(algorithmic bytes = S x (H + 4); issue-bound below the HBM roofline), the tcgen05 Gram kernels are paced by "
                    "the per-stage chain TMA -> bit-to-byte expansion -> proxy fence -> MMA -> commit (tensor pipe 19-31 % busy, "
                    "issue slots 50-62 %, no single resource saturated: profiles/r02b_k2t_gram_ncu.txt)",
            "tensor": {"kernels": "k2t_gram_n + k2t_gram_diff (tcgen05.mma kind::i8, cta_group::1, M128)", "kernel_ms": gram_ms,
                       "n_macs": macs_n, "peak_int8_macs_per_s": int8_peak,
                       "peak_source": "tools/mma_bench.cu on B200: 128 cycles per M128 N256 K32 instruction per SM",
                       "n_frac_of_int8_peak": macs_n / (km.get("k2t_gram_n", float("nan")) * 1e-3) / int8_peak}}
        del n_var, pair_macs
    except Exception as exc:
        roofline_missing = {"error": "%s: %s" % (type(exc).__name__, exc)}

    legs = {}
    variants = {}

    # =============== C3: ABBABABAwindows, strong scaling (10 M sites over the N GPUs) ===============
    if not args.no_legs:
        try:
            S3 = S // world
            spec3 = synth.SynthSpec(N_POPS, SAMPLES_PER_POP, PLOIDY, seed=SEED + 77 + 1000 * rank, miss=0.02)
            eng.synth_fill(spec3, S3)
            eng.set_pops(spec3.hap_pop(), P)
            lo3, hi3 = windows.sliding_coord_windows(np.zeros(S3, dtype=np.int32), ["chr1"], positions(S3), WIND_SIZE).ranges()
            eng.set_windows(lo3, hi3)
            counts3 = all_counts(len(lo3))
            w3 = max(max(counts3), 1)
            tab3 = PinnedArray((world * w3, 8), np.float64) if dist is not None else None

            def step3():
                if dist is not None:
                    eng.abbababa_allgather(0, 1, 2, 3, 0.5, w3, tab3.array)
                    return tab3.array
                return eng.abbababa(0, 1, 2, 3, 0.5)
            c_steps = max(3, min(args.steps, 10))
            dt3, tms3, _ = timed(step3, c_steps, 2)
            equal3 = None
            if dist is not None:
                g3 = multigpu.unpack_abba_records(multigpu.gathered_rows(tab3.array.copy(), counts3, w3))
                if rank == 0:
                    equal3, off = True, 0
                    for q in range(world):
                        sq = synth.SynthSpec(N_POPS, SAMPLES_PER_POP, PLOIDY, seed=SEED + 77 + 1000 * q, miss=0.02)
                        eng.synth_fill(sq, S3)
                        eng.set_pops(sq.hap_pop(), P)
                        lq, hq = windows.sliding_coord_windows(np.zeros(S3, dtype=np.int32), ["chr1"], positions(S3), WIND_SIZE).ranges()
                        eng.set_windows(lq, hq)
                        one = eng.abbababa(0, 1, 2, 3, 0.5)
                        keys = ("sites", "pos_sum", "ABBA", "BABA", "D", "fd", "fdM", "sitesUsed")
                        equal3 = equal3 and rows_equal(one, {k: g3[k][off:off + counts3[q]] for k in keys}, keys)
                        off += counts3[q]
                barrier()
            km3 = mean_ms(tms3)
            legs["c3"] = {"workload": "C3 ABBABABAwindows P1/P2/P3/O x 50 diploid samples, %d sites in total over %d GPU(s) "
                                      "(strong scaling), -w 50000, minData 0.5, 2 %% missing" % (S3 * world, world),
                          "value": world * S3 * c_steps / dt3, "unit": "sites/s", "ms_per_step": 1e3 * dt3 / c_steps,
                          "scaling": "strong", "sites_total": S3 * world, "kernel_ms": km3,
                          "k1_abba_GBps": S3 * (H + 4) / (km3.get("k1_abba", float("nan")) * 1e-3) / 1e9,
                          "rows_equal_single_gpu": equal3}
            if tab3 is not None:
                tab3.close()
        except Exception as exc:
            legs["c3"] = {"error": "%s: %s" % (type(exc).__name__, exc)}

        # =============== C5: freq.py + popgenWindows, 8 pops x 100 diploid samples, --windType sites -w 5000 ===============
        try:
            S5 = env_int("PG_BENCH_C5_SITES", 12_500_000)
            P5, H5 = 8, 1600
            res5 = {}
            for miss5, tag in ((0.0, "popgen"), (0.02, "popgen_missing")):
                if tag == "popgen_missing":
                    S5m = env_int("PG_BENCH_C5_MISSING_SITES", 250_000)      # the pairwise path at H = 1600 is O(H^2) per site
                else:
                    S5m = S5
                spec5 = synth.SynthSpec(P5, 100, PLOIDY, seed=SEED + 5 + 1000 * rank, miss=miss5)
                eng.synth_fill(spec5, S5m)
                eng.set_pops(spec5.hap_pop(), P5)
                lo5 = np.arange(0, S5m, 5000, dtype=np.int64)
                hi5 = np.minimum(lo5 + 5000, S5m)
                eng.set_windows(lo5, hi5)
                counts5 = all_counts(len(lo5))
                w5 = max(max(counts5), 1)
                tab5 = PinnedArray((world * w5, eng.popgen_record_width()), np.float64) if dist is not None else None

                def step5():
                    if dist is not None:
                        eng.popgen_allgather(w5, tab5.array, MIN_SITES, MIN_DATA)
                        return tab5.array
                    return eng.popgen(MIN_SITES, MIN_DATA)
                s5 = 5 if tag == "popgen" else 2
                dt5_sync, tms5, _ = timed(step5, s5, 1)
                # pipelined like the headline: exchange + read-back of batch k under the site pass of batch k+1
                def pipe5():
                    eng.popgen_gather_begin(w5, 0, MIN_SITES, MIN_DATA)
                    for k in range(1, s5):
                        eng.popgen_gather_begin(w5, k & 1, MIN_SITES, MIN_DATA)
                        eng.popgen_gather_end(w5, (k - 1) & 1)
                    return eng.popgen_gather_end(w5, (s5 - 1) & 1)
                pipe5()
                barrier()
                t0 = time.perf_counter()
                pipe5()
                dt5 = max_over_ranks(time.perf_counter() - t0)
                barrier()
                equal5 = None
                if dist is not None:
                    g5 = multigpu.unpack_device_records(multigpu.gathered_rows(tab5.array.copy(), counts5, w5), P5)
                    if rank == 0:
                        equal5, off = True, 0
                        keys = ("sites", "pos_sum", "path", "pi", "dxy", "fst")
                        for q in range(world):
                            sq = synth.SynthSpec(P5, 100, PLOIDY, seed=SEED + 5 + 1000 * q, miss=miss5)
                            eng.synth_fill(sq, S5m)
                            eng.set_pops(sq.hap_pop(), P5)
                            eng.set_windows(lo5, hi5)
                            one = eng.popgen(MIN_SITES, MIN_DATA)
                            equal5 = equal5 and rows_equal(one, {k: g5[k][off:off + counts5[q]] for k in keys}, keys)
                            off += counts5[q]
                        eng.synth_fill(spec5, S5m)
                        eng.set_pops(spec5.hap_pop(), P5)
                        eng.set_windows(lo5, hi5)
                    barrier()
                km5 = mean_ms(tms5)
                res5[tag] = {"value": world * S5m * s5 / dt5, "unit": "sites/s", "ms_per_step": 1e3 * dt5 / s5,
                             "value_sync": world * S5m * s5 / dt5_sync, "stepping": "pipelined",
                             "sites_per_gpu": S5m, "kernel_ms": km5, "rows_equal_single_gpu": equal5}
                if tag == "popgen":
                    res5[tag]["k1_popgen_GBps"] = S5m * (H5 + 4) / (km5.get("k1_popgen", float("nan")) * 1e-3) / 1e9
                    res5[tag]["k1_frac_of_hbm_peak"] = res5[tag]["k1_popgen_GBps"] / peak
                    # freq.py counts of the same shard: kernel + staged D2H of uint16 [sites x 8 x 4], slab by slab
                    slab5 = 2_000_000
                    pbuf = PinnedArray((slab5, P5, 4), np.uint16)               # pinned: written by the copy engine directly
                    buf = pbuf.array

                    def step_freq():
                        ms = 0.0
                        for s0 in range(0, S5m, slab5):
                            n = min(slab5, S5m - s0)
                            eng.site_counts(s0, n, out=buf)
                            ms += eng.last_timings().get("k1_counts", {"ms": 0.0})["ms"]
                        return ms
                    step_freq()
                    barrier()
                    t0 = time.perf_counter()
                    kms = step_freq()
                    dtf = max_over_ranks(time.perf_counter() - t0)
                    res5["freq_counts"] = {"value": world * S5m / dtf, "unit": "sites/s", "wall_ms": 1e3 * dtf,
                                           "kernel_ms": kms, "k1_counts_GBps": S5m * (H5 + 4 + 64) / (kms * 1e-3) / 1e9,
                                           "d2h_bytes": int(S5m) * P5 * 4 * 2}
                    del buf
                    pbuf.close()
                if tab5 is not None:
                    tab5.close()
            legs["c5"] = dict(res5, workload="C5 freq.py + popgenWindows: 8 pops x 100 diploid samples (H=1600), %d sites per GPU x "
                                             "%d GPU(s) (weak scaling; 8 GPUs = the 100 M-site config), --windType sites -w 5000"
                                             % (S5, world), scaling="weak")
        except Exception as exc:
            legs["c5"] = {"error": "%s: %s" % (type(exc).__name__, exc)}

        # =============== C4: distMat, 500 diploid samples x 2 M sites (single GPU) ===============
        if world == 1:
            try:
                S4 = env_int("PG_BENCH_C4_SITES", 2_000_000)
                spec4 = synth.SynthSpec(1, 500, PLOIDY, seed=SEED + 4, miss=0.02)
                eng.synth_fill(spec4, S4)
                lo4 = np.arange(0, S4, 5000, dtype=np.int64)
                hi4 = np.minimum(lo4 + 5000, S4)
                eng.set_windows(lo4, hi4)
                hap_ind = np.repeat(np.arange(500, dtype=np.int32), 2)
                out4 = PinnedArray((len(lo4), 500, 500), np.float64)           # the caller's buffer: pinned, written by the copy engine
                r4 = eng.pairdist(hap_ind, 500, False, out=out4.array)           # warm-up
                t0 = time.perf_counter()
                r4 = eng.pairdist(hap_ind, 500, False, out=out4.array)
                wall4 = time.perf_counter() - t0
                km4 = {k: v["ms"] for k, v in eng.last_timings().items()}
                # two full-shape windows (H = 1000, 5000 sites) against plain numpy (genomics.py:903-916, 934-954)
                ok4 = True
                for w in (0, len(lo4) - 1):
                    g, _ = eng.download(int(lo4[w]), int(hi4[w] - lo4[w]))
                    v = (g >= 0).astype(np.float32)
                    n = v.T @ v
                    same = sum(((g == a).astype(np.float32)).T @ (g == a).astype(np.float32) for a in range(4))
                    with np.errstate(divide="ignore", invalid="ignore"):
                        d = (n - same).astype(np.float64) / n.astype(np.float64)
                    np.fill_diagonal(d, np.nan)
                    with np.errstate(all="ignore"):
                        import warnings
                        with warnings.catch_warnings():
                            warnings.simplefilter("ignore")
                            ind = np.nanmean(d.reshape(500, 2, 500, 2), axis=(1, 3))
                    ok4 = ok4 and bool(np.allclose(r4["dist"][w], ind, rtol=1e-9, atol=1e-15, equal_nan=True))
                legs["c4"] = {"workload": "C4 distMat: 500 diploid samples (H=1000) x %d sites, -w 50000 (%d windows of 5000 sites), "
                                          "2 %% missing, individual x individual matrices to the host" % (S4, len(lo4)),
                              "value": S4 / wall4, "unit": "sites/s", "wall_ms": 1e3 * wall4, "kernel_ms": km4,
                              "kernel_ms_total": float(sum(km4.values())), "output_bytes": int(r4["dist"].nbytes),
                              "matches_numpy_on_full_shape_windows": ok4}
                del r4
                out4.close()
            except Exception as exc:
                legs["c4"] = {"error": "%s: %s" % (type(exc).__name__, exc)}

        # =============== from .geno text: the command lines themselves (single GPU) ===============
        if world == 1:
            try:
                from genomics_general_b200.cli import freq as freq_cli, popgenWindows as pgw_cli
                St = env_int("PG_BENCH_TEXT_SITES", 2_000_000)
                tdir = tempfile.mkdtemp(prefix="pg_bench_")
                t0 = time.perf_counter()
                gpath, ppath = write_workload_files(tdir, St, 0.02, SEED + 9)
                popargs = []
                for k in range(N_POPS):
                    popargs += ["-p", "pop%d" % k]
                opath = os.path.join(tdir, "out.csv")
                err_, sys.stderr = sys.stderr, open(os.devnull, "w")
                try:
                    cli_t = {}
                    for name, fn, argv in (
                            ("popgenWindows.py -w 50000 -m 100 -f phased", pgw_cli.main,
                             ["-w", str(WIND_SIZE), "-m", str(MIN_SITES), "-g", gpath, "-o", opath, "-f", "phased", "--popsFile", ppath] + popargs),
                            ("freq.py -f phased (one row of counts per site)", freq_cli.main,
                             ["-g", gpath, "-o", opath, "-f", "phased", "--popsFile", ppath] + popargs)):
                        best, phases = None, None
                        tpath = os.path.join(tdir, "timing.json")
                        for _ in range(2):
                            t1 = time.perf_counter()
                            fn(argv + ["--timing", tpath])
                            dt_ = time.perf_counter() - t1
                            if best is None or dt_ < best:
                                best = dt_
                                try:      # the command line's own --timing report: where the wall time goes
                                    tj = json.load(open(tpath))
                                    phases = {k: tj[k] for k in ("phases_s", "stage_busy_s", "total_s") if k in tj}
                                except Exception:
                                    phases = None
                        cli_t[name] = {"wall_s": best, "sites_per_s": St / best, "output_bytes": os.path.getsize(opath),
                                       "timing": phases}
                finally:
                    sys.stderr.close()
                    sys.stderr = err_
                legs["from_text"] = {"workload": "C2 shape with 2 %% missing genotypes as a %d-site .geno file (%.2f GB of text), "
                                                 "complete command lines in process: argument parsing -> device tokenizer -> "
                                                 "windows -> statistics -> rows" % (St, os.path.getsize(gpath) / 1e9),
                                     "command_lines": cli_t}
                for pth in (gpath, ppath, opath):
                    os.remove(pth)
            except Exception as exc:
                legs["from_text"] = {"error": "%s: %s" % (type(exc).__name__, exc)}

    sampler.stop()
    clocks = sampler.summary(intervals)

    if rank != 0:
        eng.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel of the headline leg (k1_site_pass, popgen mode) ----------------
    alg_bytes = S * (H + 4)
    achieved = alg_bytes / (k1_ms * 1e-3) / 1e9
    traffic = None
    try:
        traffic = json.load(open(os.path.join(REPO, "profiles", "k1_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k1_site_pass<POPGEN,4>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": k1_ms,
                "note": "the kernel only READS (4.04 GB in, a few MB out); the peak is the driver's copy figure (read + write "
                        "traffic), so a fraction slightly above 1 is a read-only stream beating a copy, not a measurement error: "
                        "ncu reports 4.050 GB of DRAM traffic for the 4.040 GB of algorithmic bytes (profiles/k1_traffic.json)",
                "missing": roofline_missing}

    # ---------------- CPU baseline: the unmodified reference command line on a bounded sample ----------------
    cpu = cpu_missing = None
    if not args.no_cpu_baseline:
        tdir = tempfile.mkdtemp(prefix="pg_cpu_")
        try:
            if have_reference():
                cpu, _ = reference_sweep(tdir, 0.0, budget_s=12.0)
                cpu_missing, _ = reference_sweep(tdir, 0.02, budget_s=12.0)
            else:
                cpu = port_sample(0.0, 4, 2000)
                cpu_missing = port_sample(0.02, 4, 2000)
        except Exception as exc:
            cpu = cpu or {"error": "%s: %s" % (type(exc).__name__, exc)}

    cfg = workload_config(args, world)
    line = {"metric": METRIC, "value": value, "unit": "sites/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * A["dt_pipe"] / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg, "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(A["launches_pipe"]), "roofline": roofline, "cpu_baseline": cpu, "kernel_ms": kernel_ms,
            "rows_equal_single_gpu": A["equal"],
            "stepping": "pipelined: the all-gather + D2H of batch k run on a side stream under the site pass of batch k+1 "
                        "(pg_popgen_gather_begin/_end); every batch's rows reach the host inside the timed region",
            "value_sync": value_sync, "ms_per_step_sync": 1e3 * A["dt"] / args.steps,
            "pipelined_rows_equal_sync": A["pipe_equal"],
            "workload_detail": {"windows_per_gpu": int(A["W"]),
                                "paths": {"failed": A["paths"][0], "closed_form_K1": A["paths"][1], "pairwise_K2": A["paths"][2]}},
            "value_missing": value_missing, "ms_per_step_missing": 1e3 * B["dt_pipe"] / m_steps,
            "value_missing_sync": value_missing_sync, "pipelined_rows_equal_sync_missing": B["pipe_equal"],
            "kernel_ms_missing": kernel_ms_missing, "roofline_missing": roofline_missing,
            "cpu_baseline_missing": cpu_missing, "rows_equal_single_gpu_missing": B["equal"],
            "paths_missing": {"failed": B["paths"][0], "closed_form_K1": B["paths"][1], "pairwise_K2": B["paths"][2]},
            "c3": legs.get("c3"), "c4": legs.get("c4"), "c5": legs.get("c5"), "from_text": legs.get("from_text"),
            "variants": variants}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"c2": A["out_rows"], "c2_missing": B["out_rows"]})
    emit(line)
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except Exception:
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        sys.exit(1)
