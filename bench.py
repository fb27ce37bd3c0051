#!/usr/bin/env python
"""bench.py -- reads/sec aligned + classified, BASELINE.json's metric.

  python bench.py --gpus N --steps K --warmup W            the CUDA engine (one rank per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU path on the host cores
  python bench.py --config single|hdr|pooled|mixed         BASELINE.json configs[1] (default) / [2] / [3] / [4]
  python bench.py ... --dump-outputs DIR                    also write the last timed step's outputs (seeded sample) as .npy

One step = one pass of the hot path over one batch of synthetic reads, every read aligned (no dedup shortcut, so
reads/s == DP problems/s):
  value : batch already resident in HBM, outputs left in HBM (device-pointer C-ABI entry)
  e2e   : the same batch through the host-pointer C-ABI call: pinned host buffers in, pinned host buffers out,
          H2D + kernel + D2H inside the timed region
Timed with CUDA events on the engine's stream, barrier + synchronize on both sides, max over ranks.
After the timed region (rank 0): the parity gate -- >= 100k reads of the timed batch re-checked against the CPU oracle on
every field a caller sees plus the count block (oracle/batch_gate.py) -- and the CPU baselines.
"""
import argparse
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

ALG_INTOPS_PER_CELL = 10                         # SURVEY.md 8(d): 5 adds, 4 max/select, 1 score lookup
GATE_READS = 1 << 17                             # reads of the timed batch checked against the oracle


# --------------------------------------------------------------------------------------------- workloads
class Workload:
    """Synthetic batch of one BASELINE.json config for one rank: refs/ref_names, packed reads (+ per-read ref_id), params."""

    def __init__(self, name, n_reads, rank):
        from crispresso2_b200 import synth
        from oracle import oracle as O
        self.name, self.n = name, n_reads
        self.flags = 0
        self.params = O.Params()
        self.ref_id = None
        rng = np.random.default_rng(1000 + rank)
        arng = np.random.default_rng(42)                                  # same amplicons on every rank
        if name == "single":
            amp = synth.random_amplicon(arng, 250)
            self.refs, self.ref_names = {"Reference": synth.amplicon_setup(amp)}, ["Reference"]
            reads = synth.synth_reads_fast(rng, amp, n_reads, 250, cut=self.refs["Reference"]["cut_point"])
            self.buf, self.off = reads.reshape(-1), np.arange(n_reads + 1, dtype=np.int64) * 250
            self.label = "synthetic %s x 250 bp reads, 1 amplicon (BASELINE.json configs[1]), every read aligned" % _fmt(n_reads)
        elif name == "hdr":
            self.refs, self.ref_names, reads = synth.hdr_workload(arng, rng, n_reads)
            self.buf, self.off = reads.reshape(-1), np.arange(n_reads + 1, dtype=np.int64) * 250
            self.params.expected_hdr_amplicon_seq = self.refs[self.ref_names[1]]["sequence"]
            from crispresso2_b200 import _lib
            self.flags = _lib.F_HDR_REF1
            self.label = "synthetic %s x 250 bp reads, 3 amplicons (HDR mode, BASELINE.json configs[2])" % _fmt(n_reads)
        elif name == "pooled":
            self.refs, self.ref_names, self.buf, self.off, self.ref_id = synth.pooled_workload(arng, rng, n_reads, 96)
            self.label = "CRISPRessoPooled synthetic: 96 amplicons (180-280 bp), %s x 250 bp reads with amplicon ids (configs[3])" % _fmt(n_reads)
        elif name == "mixed":
            amp = synth.random_amplicon(arng, 250)
            self.refs, self.ref_names = {"Reference": synth.amplicon_setup(amp)}, ["Reference"]
            self.buf, self.off = synth.mixed_length_reads(rng, amp, n_reads, 50, 300, cut=self.refs["Reference"]["cut_point"])
            self.label = "mixed-length 50-300 bp reads, %s reads, 1 amplicon (configs[4], load-balance stress)" % _fmt(n_reads)
        else:
            raise SystemExit("unknown --config %r" % name)
        lens = np.diff(self.off)
        self.max_len = int(lens.max())
        # algorithmic work of the reference algorithm on this batch (SURVEY.md 8(d)): bytes and DP cells
        I = np.array([len(self.refs[r]["sequence"]) for r in self.ref_names], dtype=np.int64)
        if self.ref_id is not None:
            cells = int((I[self.ref_id] * lens).sum())
            kept = 1
        else:
            cells = int(I.sum() * lens.sum())
            kept = 1 if len(self.ref_names) == 1 else 2                    # HDR: the winner's strings + reference 0's
        self.alg_cells = cells
        self.alg_bytes = int(lens.sum() + kept * 2 * (lens.sum() + 6 * n_reads) + 32 * n_reads)   # read + 2*aln_len per kept ref + record


def _fmt(n):
    return "%dM" % (n >> 20) if n % (1 << 20) == 0 else "%dk" % (n // 1000) if n % 1000 == 0 else str(n)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                t = [x.strip() for x in out.strip().split(",")]
                if len(t) >= 6:
                    self.rows.append(t)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# ----------------------------------------------------------------------------------------- CPU baselines
def cpu_model():
    try:
        with open("/proc/cpuinfo") as fh:
            for ln in fh:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def _ref_native():
    """The reference's own compiled Cython modules: baseline/_ref (pip-installed reference) or oracle/_ref."""
    from baseline import ref_shim
    if ref_shim.available():
        return ref_shim.native_modules()
    from oracle import oracle as O
    return O.ref_modules()


_JOB = {}


def _ref_worker(span):
    lo, hi = span
    A, R = _JOB["mods"]
    amp, gi, inc, strs, m = _JOB["amp"], _JOB["gi"], _JOB["inc"], _JOB["strs"], _JOB["matrix"]
    n = len(strs)
    t0 = time.time()
    for k in range(lo, hi):
        s1, s2, sc = A.global_align(strs[k % n], amp, matrix=m, gap_incentive=gi, gap_open=-20, gap_extend=-2)
        R.find_indels_substitutions(s1, s2, inc)
    return hi - lo, time.time() - t0


def bare_loop_steps(amp, ref, reads, cores, n_per_core, n_steps, n_warm):
    """Steps of cores x n_per_core reads through the reference's Cython global_align + find_indels_substitutions on a fork
    pool (no Python glue of process_fastq).  The sample is cycled, so every step is full; asserted."""
    import multiprocessing as mp
    mods = _ref_native()
    if mods is None:
        return None
    _JOB.update(mods=mods, amp=amp, gi=np.ascontiguousarray(ref["gap_incentive"], dtype=np.int64),
                inc=[int(v) for v in ref["include_idxs"]], strs=[r.tobytes().decode() for r in reads], matrix=mods[0].make_matrix())
    per_step = []
    with mp.get_context("fork").Pool(cores) as pool:
        pos = 0
        for step in range(n_warm + n_steps):
            spans = [(pos + c * n_per_core, pos + (c + 1) * n_per_core) for c in range(cores)]
            pos += cores * n_per_core
            t0 = time.time()
            out = pool.map(_ref_worker, spans, chunksize=1)
            dt = time.time() - t0
            done = sum(o[0] for o in out)
            if done != cores * n_per_core:
                raise RuntimeError("reference arm: step %d processed %d reads, expected %d" % (step, done, cores * n_per_core))
            if step >= n_warm:
                per_step.append((done, dt))
    return per_step


def reference_process_fastq(amp, ref, reads, n_processes):
    """The UNMODIFIED reference process_fastq (CRISPRessoCORE.py:1735-2000, installed under baseline/_ref) on a FASTQ of
    `reads`: -> (reads/s, unique reads, seconds) or None when baseline/_ref is absent."""
    from baseline import ref_shim
    if not ref_shim.available():
        return None
    import logging
    from crispresso2_b200 import synth
    CORE = ref_shim.load_core()
    from CRISPResso2 import CRISPRessoShared
    logging.getLogger("CRISPResso2").setLevel(logging.ERROR)
    for name in list(logging.root.manager.loggerDict):
        if name.startswith("CRISPResso"):
            logging.getLogger(name).setLevel(logging.ERROR)
    d = tempfile.mkdtemp(prefix="c2b_ref_")
    try:
        fq = os.path.join(d, "sample.fastq")
        synth.write_fastq(fq, reads)
        args = CRISPRessoShared.getCRISPRessoArgParser("Core").parse_args(["-r1", fq, "-a", amp])
        args.n_processes = str(n_processes)
        cache = {}
        out_fd = os.dup(1)
        try:                                                # the reference logs to stdout: keep our JSON line alone there
            os.dup2(2, 1)
            t0 = time.time()
            st, lost = CORE.process_fastq(fq, cache, ["Reference"], {"Reference": ref}, args, [], d)
            dt = time.time() - t0
        finally:
            sys.stdout.flush()
            os.dup2(out_fd, 1)
            os.close(out_fd)
        assert st["N_TOT_READS"] == len(reads)
        return {"reads_per_s": len(reads) / dt, "unique_reads": st["N_COMPUTED_ALN"] + st["N_COMPUTED_NOTALN"],
                "unique_per_s": (st["N_COMPUTED_ALN"] + st["N_COMPUTED_NOTALN"]) / dt, "seconds": dt, "reads": len(reads),
                "n_processes": n_processes}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def cpu_baseline_port(amp, ref, reads, seconds=10.0):
    """The oracle's C restatement (single thread, no Python in the loop) on a bounded sample."""
    import ctypes as C
    from oracle import oracle as O
    L = O.lib()
    m = np.ascontiguousarray(O.make_matrix())
    mask = np.zeros(len(amp) + 2, dtype=np.uint8)
    mask[ref["include_idxs"]] = 1
    gi = np.ascontiguousarray(ref["gap_incentive"], dtype=np.int64)
    n, rl = 2000, reads.shape[1]
    done, t0, chk = 0, time.time(), C.c_int64(0)
    while time.time() - t0 < seconds:
        blk = np.ascontiguousarray(reads[(done % (len(reads) - n)):(done % (len(reads) - n)) + n])
        off = np.arange(n + 1, dtype=np.int64) * rl
        L.c2o_batch_align_classify(blk.ctypes.data, off.ctypes.data, n, amp.encode(), len(amp), m.ctypes.data, m.shape[1],
                                   gi.ctypes.data, -20, -2, mask.ctypes.data, C.byref(chk))
        done += n
    dt = time.time() - t0
    return {"value": done / dt, "unit": "reads/s", "cores": 1, "kind": "port",
            "sample": "%d reads of the same workload, oracle/c2_oracle.c global_align+find_indels, 1 thread, %.1f s" % (done, dt)}


def cpu_baseline_block(amp, ref, reads, full=True):
    """cpu_baseline object: the reference's Cython loop on all cores (value) + BASELINE.md section 4's process_fastq legs."""
    cores = os.cpu_count() or 1
    n_per_core = 1500
    steps = bare_loop_steps(amp, ref, reads[:50000], cores, n_per_core, 2, 1)
    if steps is None:
        base = cpu_baseline_port(amp, ref, reads)
        base["cpu_model"] = cpu_model()
        return base
    n_done, t = sum(s[0] for s in steps), sum(s[1] for s in steps)
    out = {"value": n_done / t, "unit": "reads/s", "cores": cores, "kind": "reference", "cpu_model": cpu_model(),
           "sample": "%d reads per step x %d steps (%d per core, sample cycled), the reference's Cython global_align + "
                     "find_indels_substitutions on a fork pool, %.1f s" % (cores * n_per_core, len(steps), n_per_core, t)}
    if full:
        one = reference_process_fastq(amp, ref, reads[:16000], 1)
        if one:
            out["process_fastq_p1"] = one
            allc = reference_process_fastq(amp, ref, reads[:max(16000, min(len(reads), 400 * cores))], cores)
            out["process_fastq_pall"] = allc
        bare1 = bare_loop_steps(amp, ref, reads[:4000], 1, 4000, 1, 0)
        out["bare_loop_1core"] = {"reads_per_s": bare1[0][0] / bare1[0][1], "reads": bare1[0][0]}
    return out


def api_leg(w, eng, reads, label):
    """The call a CRISPResso maintainer binds: FASTQ file -> crispresso2_b200.core.process_fastq (CRISPRessoCORE.py:1735) ->
    core.quantify (the count block of the quantification loop, :3964-4272), wall clock, file already in the page cache.
    Nothing is skipped: native FASTQ parse + exact dedup, rc-merge weights, H2D, kernels, D2H, aln_stats, the lazy variantCache
    (one entry per aligned unique read), the count vectors re-labelled; then 2000 cache entries are materialised to price
    the lazy payloads."""
    import types
    from crispresso2_b200 import core, synth
    from oracle import oracle as O
    d = tempfile.mkdtemp(prefix="c2b_api_")
    try:
        fq = os.path.join(d, "reads.fastq")
        synth.write_fastq_fast(fq, reads)
        a = types.SimpleNamespace(**vars(w.params))
        a.use_legacy_insertion_quantification = False
        a.prime_editing_pegRNA_scaffold_seq = ""
        a.prime_editing_pegRNA_extension_seq = ""
        a.needleman_wunsch_aln_matrix_loc = "EDNAFULL"
        a.n_processes = "1"
        m = O.make_matrix()
        best = None
        for rep in range(3):                                   # first pass warms the page cache, allocations and the engine
            cache = {}
            t0 = time.perf_counter()
            st, lost = core.process_fastq(fq, cache, w.ref_names, w.refs, a, [], d, engine=eng, aln_matrix=m)
            block = core.quantify(cache)
            vec = {r: block.vectors(r) for r in w.ref_names}
            cc = block.class_counts()
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, dict(core.last_timings), st, len(cache), len(lost))
        dt, tm, st, n_al, n_lost = best
        t0 = time.perf_counter()
        k = 0
        for seq, v in cache.items():
            _ = v["variant_" + v["best_match_name"]]["ref_positions"]
            k += 1
            if k >= 2000:
                break
        t_mat = (time.perf_counter() - t0) / max(1, k)
        assert st["N_TOT_READS"] == len(reads) and sum(cc.values()) > 0 and len(vec) == len(w.ref_names)
        nu = tm.get("n_unique", n_al + n_lost)
        return {"workload": label, "reads": int(len(reads)), "unique_reads": int(nu), "seconds": dt, "reads_per_s": len(reads) / dt,
                "unique_per_s": nu / dt, "fastq_bytes": os.path.getsize(fq), "fastq_MB_per_s": os.path.getsize(fq) / dt / 1e6,
                "stages_s": {k2: round(v2, 4) for k2, v2 in tm.items() if isinstance(v2, float)},
                "materialise_us_per_variant": t_mat * 1e6, "aligned_unique": n_al, "not_aligned_unique": n_lost,
                "call": "core.process_fastq(fastq, variantCache, ref_names, refs, args, [], outdir) + core.quantify(variantCache); best of 3"}
    finally:
        import shutil
        shutil.rmtree(d, ignore_errors=True)


def _ingest_device():
    return int(os.environ.get("LOCAL_RANK", "0"))


def ingest_leg(reads):
    """FASTQ front end alone (SURVEY.md 8f rank 1): native parse + exact de-duplication (c2b_fastq_dedup: what feeds the kernels)
    and the native quality filter (c2b_fastq_filter), on the timed batch written as plain text and -- a 256k-read slice -- as
    gzip.  Wall clock, file in the page cache, best of 3."""
    import gzip
    import shutil
    from crispresso2_b200 import fastq, filter_fastqs, synth
    d = tempfile.mkdtemp(prefix="c2b_ing_")
    out = {}
    try:
        plain = os.path.join(d, "r.fastq")
        synth.write_fastq_fast(plain, reads)
        sub = reads[:1 << 18]
        small = os.path.join(d, "s.fastq")
        synth.write_fastq_fast(small, sub)
        gz = os.path.join(d, "s.fastq.gz")
        with open(small, "rb") as fi, gzip.open(gz, "wb", compresslevel=1) as fo:
            shutil.copyfileobj(fi, fo, 1 << 22)

        bgz = os.path.join(d, "s_blocked.fastq.gz")
        with open(small, "rb") as fi, open(bgz, "wb") as fo:
            fo.write(synth.bgzf_bytes(fi.read()))

        def best(fn, reps=3):
            t = []
            for _ in range(reps):
                t0 = time.perf_counter()
                r = fn()
                t.append(time.perf_counter() - t0)
            return min(t), r

        for name, path, n in (("dedup_plain", plain, len(reads)), ("dedup_gzip", gz, len(sub)), ("dedup_blocked_gzip", bgz, len(sub))):
            dt, dd = best(lambda: fastq.dedup_file(path))
            assert dd.n_reads == n
            out[name] = {"reads": n, "unique": int(len(dd.counts)), "seconds": dt, "reads_per_s": n / dt,
                         "file_MB_per_s": os.path.getsize(path) / dt / 1e6}
        for name, path, n in (("dedup_gpu_plain", plain, len(reads)), ("dedup_gpu_gzip", gz, len(sub)), ("dedup_gpu_blocked_gzip", bgz, len(sub))):
            # the same front end on the GPU (c2b_fastq_dedup_gpu): file bytes over PCIe once, parse + exact dedup on the device
            dt, dg = best(lambda: fastq.dedup_file(path, device=_ingest_device()))
            hd = fastq.dedup_file(path)
            assert dg.n_reads == n and np.array_equal(dg.off, hd.off) and np.array_equal(dg.buf, hd.buf) and np.array_equal(dg.counts, hd.counts)
            out[name] = {"reads": n, "unique": int(len(dg.counts)), "seconds": dt, "reads_per_s": n / dt,
                         "file_MB_per_s": os.path.getsize(path) / dt / 1e6, "equals_host_front_end": True}
        for name, path, n in (("filter_plain", plain, len(reads)), ("filter_gzip_in_out", gz, len(sub))):
            dst = os.path.join(d, "f_" + os.path.basename(path))
            dt, r = best(lambda: filter_fastqs.filterFastqs(fastq_r1=path, fastq_r1_out=dst, min_av_read_qual=30, min_bp_qual_or_N=20), reps=2)
            out[name] = {"reads": n, "kept": int(r[1]), "seconds": dt, "reads_per_s": n / dt, "file_MB_per_s": os.path.getsize(path) / dt / 1e6}
        return out
    finally:
        shutil.rmtree(d, ignore_errors=True)


def reference_arm(args, emit):
    """--impl reference: the reference's own Cython global_align + find_indels_substitutions (compiled from /root/reference,
    unmodified) on all host cores, on a bounded sample per step; falls back to the oracle port when neither baseline/_ref
    nor oracle/_ref travelled."""
    cores = os.cpu_count() or 1
    w = Workload("single", 200_000, 0)
    amp, ref = w.refs["Reference"]["sequence"], w.refs["Reference"]
    reads = w.buf.reshape(-1, 250)
    n_per_core = 600                                             # ~0.6 ms per read -> ~0.4 s per core per step
    steps = bare_loop_steps(amp, ref, reads, cores, n_per_core, args.steps, args.warmup)
    if steps is not None:
        kind = "reference"
        sample = ("%d reads per step (%d per core, 200k-read sample cycled; every step asserted full), the reference's Cython "
                  "global_align + find_indels_substitutions via fork pool" % (cores * n_per_core, n_per_core))
    else:
        base = cpu_baseline_port(amp, ref, reads, seconds=10.0)
        steps = [(base["value"] * 1.0, 1.0)]
        kind, cores, sample = "port", 1, base["sample"]
    n_done = sum(p[0] for p in steps)
    t = sum(p[1] for p in steps)
    val = n_done / t
    cb = {"value": val, "unit": "reads/s", "cores": cores, "kind": kind, "sample": sample, "cpu_model": cpu_model()}
    if kind == "reference" and args.gpus == 1 and not args.no_cpu_baseline:
        one = reference_process_fastq(amp, ref, reads[:16000], 1)
        if one:
            cb["process_fastq_p1"] = one
            cb["process_fastq_pall"] = reference_process_fastq(amp, ref, reads[:max(16000, min(len(reads), 400 * cores))], cores)
    line = {"impl": "reference", "metric": "reads/sec aligned+classified (250 bp, single amplicon)", "value": val,
            "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * t / max(1, len(steps)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": "synthetic 1M x 250 bp reads, 1 amplicon (bounded sample per step)"},
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="single", choices=["single", "hdr", "pooled", "mixed"])
    ap.add_argument("--reads", type=int, default=1 << 20, help="reads per GPU per step (weak scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gate", action="store_true", help="skip the oracle parity gate (profiling runs only)")
    ap.add_argument("--edit-cap", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-api", action="store_true", help="skip the process_fastq (api) leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    # stdout carries the ONE JSON line and nothing else: libraries that write to fd 1 (NCCL's version banner, the reference's
    # logger) go to stderr for the whole run; the line is written to the saved descriptor at the end
    sys.stdout.flush()
    real_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def emit(line):
        real_out.write(json.dumps(line) + "\n")
        real_out.flush()

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, emit)
        return 0

    import torch
    import torch.distributed as dist
    from crispresso2_b200 import _lib, dist as cdist
    from crispresso2_b200.engine import Engine
    from oracle import oracle as O

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if args.warmup < 3:
        args.warmup = 3

    n = args.reads
    w = Workload(args.config, n, rank)
    eng = Engine(local)
    P = w.params
    eng.configure(w.refs, w.ref_names, O.make_matrix(), P.needleman_wunsch_gap_open, P.needleman_wunsch_gap_extend,
                  P.aln_seed_count, P.aln_seed_min, w.flags, "ACGTN", args.edit_cap)
    W = eng.string_width(w.max_len)
    R = 1 if w.ref_id is not None else len(w.ref_names)
    L = eng.L
    stream = torch.cuda.ExternalStream(L.c2b_stream(eng.h), device=dev)

    # ---- device-resident buffers (value leg) -------------------------------------------------------
    d_reads = torch.from_numpy(np.ascontiguousarray(w.buf)).to(dev)
    d_off = torch.from_numpy(w.off).to(dev)
    d_rid = torch.from_numpy(w.ref_id).to(dev) if w.ref_id is not None else None
    d_recs = torch.empty(n * 16, dtype=torch.uint8, device=dev)
    d_alns = torch.empty(n * R * 32, dtype=torch.uint8, device=dev)
    d_str = torch.empty(n * R * 2 * W, dtype=torch.uint8, device=dev)
    d_ed = torch.empty(n * R * args.edit_cap * 8, dtype=torch.uint8, device=dev)
    d_ord = None
    if len(np.unique(np.diff(w.off))) > 1 or w.ref_id is not None:      # mixed lengths / amplicons: equal ones adjacent (pairing order)
        key = np.diff(w.off) if w.ref_id is None else w.ref_id.astype(np.int64) * 1024 + np.diff(w.off)
        d_ord = torch.from_numpy(np.argsort(key, kind="stable").astype(np.int32)).to(dev)
        L.c2b_set_pair_order(eng.h, d_ord.data_ptr())
    torch.cuda.synchronize(dev)

    def step_device():
        rc = L.c2b_align_batch_device(eng.h, d_reads.data_ptr(), d_off.data_ptr(), n, w.max_len, None, None,
                                      d_rid.data_ptr() if d_rid is not None else None,
                                      d_recs.data_ptr(), d_alns.data_ptr(), d_str.data_ptr(), d_ed.data_ptr())
        if rc != 0:
            raise RuntimeError(L.c2b_last_error(eng.h).decode())
        if world > 1:                       # merge of the count block: the path's only exchange (NCCL, NVLink)
            cdist.allreduce_counts(eng)

    def barrier():
        if world > 1:
            dist.barrier()
        eng.sync()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        eng.counts_reset()
        step_device()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    launches0 = eng.launch_count()
    kernel_ms = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.counts_reset()
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
        kernel_ms.append(eng.last_kernel_ms())         # CUDA events around the kernel(s) on their own stream
    ev1.record(stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    pair_items, single_items = eng.path_counts()
    L.c2b_set_pair_order(eng.h, None)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, args.steps, n, R, W, args.edit_cap, d_recs, d_alns, d_str, d_ed)

    recs = np.frombuffer(d_recs.cpu().numpy().tobytes(), dtype=_lib.REC_DTYPE)
    alns = np.frombuffer(d_alns.cpu().numpy().tobytes(), dtype=_lib.ALN_DTYPE).reshape(n, R)
    aligned_frac = float((recs["best_score_milli"] > 0).mean())

    # ---- parity gate on this very batch: the first GATE_READS reads against the oracle, every field + count block ----
    gate = {"reads": 0, "ok": None}
    if rank == 0 and not args.no_gate:
        gate = parity_gate(eng, w, args, recs, alns, d_str, d_ed, W, R, dev)

    # ---- end-to-end leg: host buffers through c2b_align_batch --------------------------------------
    import ctypes as C

    def pinned(nbytes, dtype=np.uint8):
        p = L.c2b_host_alloc(nbytes)
        if not p:
            raise MemoryError("c2b_host_alloc")
        return np.frombuffer((C.c_uint8 * nbytes).from_address(p), dtype=np.uint8).view(dtype), p

    nb = int(w.off[-1])
    NW = L.c2b_ops_words(eng.h, w.max_len)
    h_reads, p1 = pinned(nb)
    h_reads[:] = w.buf
    h_off, p2 = pinned((n + 1) * 8, np.int64)
    h_off[:] = w.off
    h_recs, p3 = pinned(n * 16)
    h_alns, p4 = pinned(n * R * 32)
    h_ops, p5 = pinned(n * R * NW * 8)
    h_meta, p8 = pinned(n * R * 4)
    h_ed, p6 = pinned(n * R * args.edit_cap * 8)
    h_rid, p7 = (None, None)
    if w.ref_id is not None:
        h_rid, p7 = pinned(n * 4, np.int32)
        h_rid[:] = w.ref_id
    h2d = nb + (n + 1) * 8 + (n * 4 if w.ref_id is not None else 0)

    def step_e2e():
        # the compact form of the host-buffer call: op streams + meta words instead of the spelled-out strings
        rc = L.c2b_align_batch_compact(eng.h, h_reads.ctypes.data, h_off.ctypes.data, n, None, None,
                                       h_rid.ctypes.data if h_rid is not None else None, h_recs.ctypes.data,
                                       h_alns.ctypes.data, h_ops.ctypes.data, h_meta.ctypes.data, h_ed.ctypes.data)
        if rc != 0:
            raise RuntimeError(L.c2b_last_error(eng.h).decode())
        if world > 1:
            cdist.allreduce_counts(eng)

    e2e_steps = max(2, args.e2e_steps)
    step_e2e()
    step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(e2e_steps):
        step_e2e()
    e1.record(stream)
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    h_al = np.frombuffer(h_alns.tobytes(), dtype=_lib.ALN_DTYPE).reshape(n, R)
    e2e_gate = bool((h_al["n_match"] == alns["n_match"]).all() and (h_al["aln_len"] == alns["aln_len"]).all()
                    and (h_al["n_sub_all"] == alns["n_sub_all"]).all())
    # ... and the strings rebuilt on the host from the compact outputs equal the ones the device-resident leg left in HBM
    if rank == 0:
        G = min(GATE_READS, n)
        exp = np.zeros((G, R, 2, W), dtype=np.uint8)
        rc = L.c2b_expand_batch(eng.h, h_reads.ctypes.data, h_off.ctypes.data, G, h_rid.ctypes.data if h_rid is not None else None,
                                h_ops.ctypes.data, h_meta.ctypes.data, w.max_len, exp.ctypes.data, 0)
        t_str = d_str[: G * R * 2 * W].cpu().numpy().reshape(G, R, 2, W)
        cols = np.arange(W)[None, None, None, :] >= (W - alns[:G]["aln_len"].astype(np.int64))[:, :, None, None]
        has = (alns[:G]["aln_len"] > 0)[:, :, None, None]
        e2e_gate = e2e_gate and rc == 0 and bool(((exp == t_str) | ~(cols & has)).all())
    # only the first Wt/32 op words of every slot cross PCIe (Wt = the chunk's widest alignment, rounded to 32)
    Wt = min(W, (int(h_al["aln_len"].max()) + 31) & ~31)
    d2h = n * 16 + n * R * 32 + n * R * (Wt // 32) * 8 + n * R * 4 + n * R * args.edit_cap * 8
    # secondary: the same batch with the spelled-out strings coming back (c2b_align_batch), fewer steps
    h_str, p9 = pinned(n * R * 2 * W)

    def step_e2e_strings():
        rc = L.c2b_align_batch(eng.h, h_reads.ctypes.data, h_off.ctypes.data, n, None, None,
                               h_rid.ctypes.data if h_rid is not None else None, h_recs.ctypes.data,
                               h_alns.ctypes.data, h_str.ctypes.data, h_ed.ctypes.data)
        if rc != 0:
            raise RuntimeError(L.c2b_last_error(eng.h).decode())
        if world > 1:
            cdist.allreduce_counts(eng)

    step_e2e_strings()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for _ in range(3):
        step_e2e_strings()
    s1.record(stream)
    barrier()
    e2s_ms = s0.elapsed_time(s1)
    d2h_strings = n * 16 + n * R * 32 + n * R * 2 * Wt + n * R * args.edit_cap * 8
    if sampler:                                  # sampled across the timed regions (device-resident and end-to-end)
        sampler.stop_flag = True
        sampler.join(timeout=3)
    for p in (p1, p2, p3, p4, p5, p6, p7, p8, p9):
        if p:
            L.c2b_host_free(p)

    # ---- reduce over ranks ----------------------------------------------------------------------------
    t = torch.tensor([dev_ms, e2e_ms, float(np.mean(kernel_ms)), e2s_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, k_ms, e2s_ms = [float(x) for x in t.cpu()]
    total_reads = n * world
    value = total_reads * args.steps / (dev_ms / 1000.0)
    e2e_val = total_reads * e2e_steps / (e2e_ms / 1000.0)

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peaks = json.load(fh)
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = w.alg_bytes / (k_ms / 1000.0) / 1e9
        traffic, executed = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and args.config == "single":
            try:
                with open(tpath) as fh:
                    tj = json.load(fh)
                traffic, executed = tj.get("dram_bytes_per_launch"), tj.get("executed")
            except Exception:
                traffic = None
        clocks = sampler.summary() if sampler else {}
        sm_clk = clocks.get("sm_mhz") or 1965
        int_peak = 148 * 128 * sm_clk * 1e6            # int32 lanes/clk/SM (ALU + FMA pipes, B300_MICROARCH.md) x clock
        alg_ops = w.alg_cells * ALG_INTOPS_PER_CELL
        metric = {"single": "reads/sec aligned+classified (250 bp, single amplicon)",
                  "hdr": "reads/sec aligned+classified (250 bp, 3 amplicons, HDR mode)",
                  "pooled": "reads/sec aligned+classified (250 bp, 96 amplicons, Pooled)",
                  "mixed": "reads/sec aligned+classified (50-300 bp, single amplicon)"}[args.config]
        line = {
            "metric": metric, "value": value, "unit": "reads/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": w.label,
                       "reads_per_gpu_per_step": n, "parallelism": "read-shard x%d" % world,
                       "l2": "inputs+outputs per step (%.2f GB) exceed the 126 MB L2" % ((h2d + d2h) / 1e9),
                       "edit_cap": args.edit_cap, "aligned_fraction": aligned_frac,
                       "packed_pair_items": pair_items, "single_items": single_items, "band_reruns": eng.band_reruns(),
                       "ring_pairs": eng.ring_counts()[0], "ring_fallbacks": eng.ring_counts()[1],
                       "parity_gate": bool(gate["ok"] and e2e_gate) if gate["ok"] is not None else None,
                       "parity_gate_detail": gate},
            "e2e": {"value": e2e_val, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                    "api": "c2b_align_batch_compact: pinned host buffers in; records, op streams, meta words and edit lists out "
                           "(aligned strings rebuilt on the host by c2b_expand_batch: checked equal to the device-resident leg's)",
                    "pipeline": "chunks of up to 256 Ki reads (a small first and last one) through two staging sets: H2D | ALIGN tier 1, tier 2, CLASSIFY, general kernel | D2H",
                    "with_strings": {"value": total_reads * 3 / (e2s_ms / 1000.0), "ms_per_step": e2s_ms / 3, "steps": 3,
                                     "d2h_bytes_per_step": d2h_strings, "api": "c2b_align_batch (two W-byte strings per slot)"}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": "measured" if peaks else "fallback",
                         "kernel": "c2b_align_kernel + c2b_classify_kernel + c2b_align_classify_kernel (left-overs), one batch", "kernel_ms": k_ms, "alg_bytes_per_launch": w.alg_bytes,
                         "secondary_int32": {"alg_ops_per_launch": alg_ops,
                                             "note": "alg_*: ops of the reference's full-matrix algorithm (10 per DP cell), a rate of USEFUL work, not a "
                                                     "utilisation: the banded DP evaluates a fraction of the cells.  executed_*: from the ncu capture "
                                                     "under profiles/ (warp instructions x 32 lanes on the issue slots), the utilisation figure",
                                             "alg_tops": alg_ops / (k_ms / 1000.0) / 1e12,
                                             "peak_tops_at_observed_clock": int_peak / 1e12,
                                             "alg_frac_of_peak": alg_ops / (k_ms / 1000.0) / int_peak,
                                             "executed": executed}},
            "clocks": clocks,
        }
        if not args.no_api and world == 1 and args.config == "single":
            from crispresso2_b200 import synth as _synth
            rd = w.buf.reshape(-1, 250)
            amp_seq = w.refs["Reference"]["sequence"]
            uniq = _synth.synth_reads_fast(np.random.default_rng(77), amp_seq, n, 250, sub_rate=0.02, cut=w.refs["Reference"]["cut_point"])
            line["api"] = {"process_fastq": api_leg(w, eng, rd, "the timed batch as a FASTQ file (%s reads)" % _fmt(n)),
                           "process_fastq_all_unique": api_leg(w, eng, uniq, "all-unique variant (substitution rate 0.02), %s reads" % _fmt(n))}
            import contextlib
            with contextlib.redirect_stdout(sys.stderr):      # filterFastqs prints its completion line, like the reference
                line["api"]["ingest"] = ingest_leg(rd)
            # paired-end merge mode (SURVEY 8f rank 3): the reference's process_paired_fastq against paired.process_paired_fastq
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import paired_bench
            line["api"]["paired_merge"] = paired_bench.run(5000, local)
        if not args.no_cpu_baseline and world == 1 and args.config == "single":
            line["cpu_baseline"] = cpu_baseline_block(w.refs["Reference"]["sequence"], w.refs["Reference"], w.buf.reshape(-1, 250))
        elif not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_generic(w)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


DUMP_READS = 1 << 15                             # seeded sample of the timed batch written by --dump-outputs
DUMP_STRING_READS = 1 << 10                      # ... and the part of it whose aligned strings are written
DUMP_LIMIT = 64 << 20


def dump_outputs(dirpath, eng, steps, n, R, W, cap, d_recs, d_alns, d_str, d_ed):
    """--dump-outputs: what a caller of c2b_align_batch_device receives after the last timed step, on a fixed seeded sample of
    the batch's reads (the batch itself is seeded too, so two builds can be compared file for file): every field of the read
    records and of the per-amplicon alignment records, the edit lists and the aligned strings with the unused entries zeroed,
    and the count block divided by the number of timed steps (it accumulates over them).  float64 where a field can exceed
    float32's exact integers."""
    from crispresso2_b200 import _lib
    os.makedirs(dirpath, exist_ok=True)
    idx = np.sort(np.random.default_rng(20240).choice(n, size=min(n, DUMP_READS), replace=False))
    recs = np.frombuffer(d_recs.cpu().numpy().tobytes(), dtype=_lib.REC_DTYPE)[idx]
    alns = np.frombuffer(d_alns.cpu().numpy().tobytes(), dtype=_lib.ALN_DTYPE).reshape(n, R)[idx]
    edits = np.frombuffer(d_ed.cpu().numpy().tobytes(), dtype=_lib.EDIT_DTYPE).reshape(n, R, cap)[idx]
    sidx = idx[:DUMP_STRING_READS]
    strs = d_str.cpu().numpy().reshape(n, R, 2, W)[sidx].astype(np.float32)
    out = {"read_index": idx.astype(np.float64)}
    for f in _lib.REC_DTYPE.names:
        out["rec_" + f] = recs[f].astype(np.float64)
    for f in _lib.ALN_DTYPE.names:
        out["aln_" + f] = alns[f].astype(np.float64)
    used = np.arange(cap)[None, None, :] < np.minimum(alns["n_edits"], cap)[:, :, None]
    for f in ("a", "b", "type", "in_window", "base"):
        out["edit_" + f] = np.where(used, edits[f], 0).astype(np.float32)
    cols = np.arange(W)[None, None, None, :] >= (W - alns["aln_len"][:len(sidx)].astype(np.int64))[:, :, None, None]
    out["strings"] = np.where(cols, strs, 0).astype(np.float32)
    out["string_read_index"] = sidx.astype(np.float64)
    out["counts"] = eng.counts_raw().astype(np.float64) / steps
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    for name, a in out.items():
        np.save(os.path.join(dirpath, name + ".npy"), a)


def cpu_baseline_generic(w):
    """Configs other than the single amplicon: the oracle's per-read path (C-backed global_align / find_indels, Python glue)
    over a fork pool on a bounded sample."""
    from oracle import batch_gate as BG
    n = min(w.n, 200 * (os.cpu_count() or 1), 65536)
    t0 = time.time()
    summ = BG.time_oracle(w.buf, w.off, w.refs, w.ref_names, w.params, w.ref_id, n)
    dt = time.time() - t0
    return {"value": n / summ["seconds"], "unit": "reads/s", "cores": summ["workers"], "kind": "port", "cpu_model": cpu_model(),
            "sample": "%d reads of the same workload, oracle.new_variant (C global_align + find_indels, Python glue) on a fork pool, "
                      "%.1f s (%.1f s with start-up)" % (n, summ["seconds"], dt)}


def parity_gate(eng, w, args, recs, alns, d_str, d_ed, W, R, dev):
    """First GATE_READS reads of the timed batch: (1) re-run alone with an edit cap that cannot overflow -- records and
    strings must equal the timed run's bit for bit; (2) every field of every read against the oracle (oracle/batch_gate.py);
    (3) the count block of that sub-batch against the oracle's quantification loop."""
    from crispresso2_b200 import _lib
    from oracle import batch_gate as BG
    from oracle import oracle as O
    G = min(GATE_READS, w.n)
    t0 = time.time()
    off = w.off[:G + 1]
    buf = w.buf[:off[-1]]
    rid = w.ref_id[:G] if w.ref_id is not None else None
    cap0 = eng.edit_cap
    eng.set_edit_cap(64)
    eng.counts_reset()
    res = eng.align_packed(buf, off, ref_id=rid)
    block = eng.counts()
    over = int(((res.recs["status"] & _lib.ST_EDIT_OVERFLOW) != 0).sum())
    eng.set_edit_cap(cap0)
    # (1) the timed run's outputs for the same reads
    t_str = d_str[: G * R * 2 * W].cpu().numpy().reshape(G, R, 2, W)
    ta, ga = alns[:G], res.alns
    same = True
    for f in _lib.ALN_DTYPE.names:
        if f in ("n_edits", "status"):
            continue
        same = same and bool((ta[f] == ga[f]).all())
    keep = np.uint8(0xff ^ _lib.ST_EDIT_OVERFLOW)
    same = same and bool(((ta["status"] & keep) == (ga["status"] & keep)).all())
    for f in ("winner_mask", "best_score_milli", "best_ref", "n_winners", "ambiguous"):
        same = same and bool((recs[:G][f] == res.recs[f]).all())
    cols = np.arange(W)[None, None, None, :] >= (W - ga["aln_len"].astype(np.int64))[:, :, None, None]
    same = same and bool(((t_str == res.strings) | ~cols).all())
    # (2) + (3)
    summ, quant = BG.run(buf, off, w.refs, w.ref_names, w.params, O.make_matrix(), res.recs, res.alns, res.strings, res.edits,
                         res.W, flags=w.flags, ref_id=rid)
    if rid is None:
        bad_counts = BG.compare_block(block, quant[None], w.ref_names, hdr=bool(w.flags & _lib.F_HDR_REF1))
    else:
        bad_counts = []
        for name, q in quant.items():
            bad_counts += BG.compare_block(block, q, [name], per_amplicon=True)
    ok = same and summ["n_bad"] == 0 and not bad_counts and over == 0
    return {"reads": G, "ok": bool(ok), "timed_equals_gate_run": bool(same), "reads_differing_from_oracle": summ["n_bad"],
            "examples": [str(b) for b in summ["bad"][:3]], "oracle_undefined_skipped": summ["n_skipped"],
            "count_block_mismatches": [str(b) for b in bad_counts[:5]], "edit_overflow_at_cap_64": over,
            "fields": "aln_scores, ref_aln_details (both aligned strings + score per reference), best_match_score, aln_ref_names, "
                      "class_name, best_match_name, all 31 payload slots; count block: every vector / counter / Counter",
            "oracle_workers": summ["workers"], "seconds": round(time.time() - t0, 1)}


if __name__ == "__main__":
    sys.exit(main())
