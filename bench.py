#!/usr/bin/env python
"""bench.py -- the headline metric of BASELINE.json on synthetic data:
reads/s mapped for 2x150 bp paired-end reads against a 3.1 Gb human-scale synthetic reference whose UFI index
(27 GB hash table + 3.1 GB sequence) is resident in each B200's HBM.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's own CPU path (oracle/_ref/urmap) on the host cores

A "step" is one pass of the hot path (probe kernel + search kernels) over one batch of `--pairs-per-step` read
pairs per GPU.  `value` is measured with the inputs already resident in HBM: K steps issued back to back, device time
between two CUDA events that bracket them; `e2e` goes through the C-ABI with pinned host buffers, H2D and D2H inside the
timed region, six batch slots in flight.  Weak scaling: every rank maps its own batches; the only collective is the
NCCL broadcast of the index at start-up.

At N = 1 the line also carries `configs`: the other BASELINE.json configurations (single-end, high-divergence reads,
250-base reads drawn from the segmental duplications / tandem repeats of the same reference), each with its kernel
times, work counters and the identity of the drop-in's SAM file with the reference binary's on >= 1 M reads.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from

import numpy as np


_OUT = sys.stdout


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.active = False
        self.proc = None
        self.th = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        for line in self.proc.stdout:
            if self.active:
                self.samples.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_json(name):
    try:
        return json.load(open(os.path.join(ROOT, name)))
    except Exception:
        return {}


# The other BASELINE.json configurations (the headline one, configs[2], is the main workload of the line).  units = reads
# (single-end) or pairs per step; every batch is larger than L2.  `enrich`: share of the reads drawn from the segmental
# duplications / tandem repeats of the reference.
EXTRA_CONFIGS = [
    dict(key="c2_se150", baseline_config=1, paired=False, read_len=150, sub=0.01, indel=0.001, enrich=0.0, units=1_000_000,
         what="single-end 150 bp, 1% subs + 0.1% indels"),
    dict(key="c4_se150_div", baseline_config=3, paired=False, read_len=150, sub=0.05, indel=0.01, enrich=0.0, units=1_000_000,
         what="single-end 150 bp, 5% subs + 1% indels (gapped Viterbi path on most reads)"),
    dict(key="c4_pe150_div", baseline_config=3, paired=True, read_len=150, sub=0.05, indel=0.01, enrich=0.0, units=500_000,
         what="paired-end 2x150 bp, 5% subs + 1% indels"),
    dict(key="c5_se250_rep", baseline_config=4, paired=False, read_len=250, sub=0.01, indel=0.001, enrich=0.5, units=1_000_000,
         what="single-end 250 bp, half of the reads from segmental duplications / tandem repeats"),
    dict(key="c5_pe250_rep", baseline_config=4, paired=True, read_len=250, sub=0.01, indel=0.001, enrich=0.5, units=500_000,
         what="paired-end 2x250 bp, half of the pairs from segmental duplications / tandem repeats"),
]


def build_workload(args, rank, world, device):
    """Genome + UFI index in HBM on every rank (rank 0 builds on its GPU, NCCL broadcast to the others)."""
    import torch

    from urmap_b200 import dist as D
    from urmap_b200 import gpu_synth, index_build
    meta, seq, blob = None, None, None
    t0 = time.time()
    if rank == 0:
        human = args.genome_len >= 100_000_000
        # the device builder does not reproduce lists the reference would truncate (it reports them): should the
        # repeat-rich genome ever produce one, fall back to fewer injected repeats rather than to a 10-minute host build
        for segdup, tandem in ((args.segdup_frac, args.tandem_frac), (args.segdup_frac, 0.0), (0.0, 0.0)):
            regions = []
            seq = blob = None
            torch.cuda.empty_cache()
            seq, names, lens, offsets, sds = gpu_synth.make_seqdata(args.genome_len, device, seed=12345,
                                                                    n_contigs=24 if human else 3, human_ratios=human,
                                                                    repeat_frac=0.10, n_runs=3, segdup_frac=segdup,
                                                                    tandem_frac=tandem, regions_out=regions)
            slot_count = index_build.slot_count_for(names, lens)
            torch.cuda.synchronize()
            log(f"genome {args.genome_len:,} bp in {len(names)} contigs generated in {time.time() - t0:.1f}s; "
                f"SeqDataSize {sds:,}; SlotCount {slot_count:,}; {len(regions)} segmental-duplication / tandem-repeat regions")
            blob = torch.empty(5 * slot_count + 16, dtype=torch.uint8, device=device)
            torch.cuda.empty_cache()
            st = index_build.build_index_device(seq.data_ptr(), sds, slot_count, blob.data_ptr())
            log(f"UFI built on the GPU: {st}")
            if not st["truncated"]:
                break
            log(f"WARNING: {st['truncated']} list(s) would be truncated with segdup {segdup} / tandem {tandem}: retrying with less")
        if st["truncated"]:
            raise RuntimeError("index has lists the reference would truncate: use the sequential builder")
        meta = {"word_length": 24, "max_ix": 32, "seq_data_size": sds, "slot_count": slot_count, "names": names,
                "lens": lens, "offsets": offsets, "seq_alloc": seq.numel(), "blob_alloc": blob.numel(),
                "build_seconds": st["seconds"], "indexed": st["indexed"], "regions": regions,
                "segdup_frac": segdup, "tandem_frac": tandem}
    t1 = time.time()
    meta, seq, blob = D.broadcast_index(meta, seq, blob, device)
    if world > 1:
        torch.cuda.synchronize()
        log(f"rank {rank}: index broadcast over NCCL in {time.time() - t1:.2f}s")
    return meta, seq, blob


def make_batches(meta, seq, device, nb, units, paired, read_len, sub, indel, seed0, enrich=0.0):
    """nb distinct batches of reads / read pairs, as pinned host numpy arrays: (h1, h2, a1, a2, offs)."""
    import torch

    from urmap_b200 import gpu_synth
    B, RL = units, read_len
    offs = (np.arange(B + 1, dtype=np.uint32) * RL)
    regions = None
    if enrich > 0 and meta.get("regions"):
        regions = gpu_synth.regions_tensor(meta["regions"], device)
    pad = 40 if indel <= 0.002 else 60
    out = []
    for k in range(nb):
        seed = seed0 + k
        kw = dict(regions=regions, enrich=enrich) if regions is not None else {}
        if not paired:
            r1 = gpu_synth.sim_se(seq, meta["lens"], meta["offsets"], B, device, RL, sub, indel, seed=seed, pad=pad, **kw)
            r2 = None
        else:
            r1, r2 = gpu_synth.sim_pe(seq, meta["lens"], meta["offsets"], B, device, RL, sub, indel, seed=seed, pad=pad, **kw)
        h1 = torch.empty(r1.shape, dtype=torch.uint8, pin_memory=True)
        h1.copy_(r1)
        h2 = None
        if r2 is not None:
            h2 = torch.empty(r2.shape, dtype=torch.uint8, pin_memory=True)
            h2.copy_(r2)
        torch.cuda.synchronize()
        out.append((h1, h2, h1.numpy().reshape(-1), None if h2 is None else h2.numpy().reshape(-1), offs))
        del r1, r2
    torch.cuda.empty_cache()
    return out


def write_ufi_file(path, meta, seq, blob):
    from urmap_b200 import index_build
    CH = 1 << 28

    def chunks(t, n):
        for o in range(0, n, CH):
            yield t[o:min(n, o + CH)].cpu().numpy().tobytes()

    index_build.write_ufi(path, meta["names"], meta["lens"], meta["offsets"], meta["seq_data_size"], meta["slot_count"],
                          chunks(blob, 5 * meta["slot_count"]), chunks(seq, meta["seq_data_size"]))


def write_fastq(path, arr, n, RL, label, suffix, mode="wb"):
    """@<label><i><suffix>, bases, '+', constant quality 'I' -- written as one 2-D byte array per label width."""
    lab = label.encode()
    with open(path, mode) as f:
        lo = 0
        width = 1
        while lo < n:
            hi = min(n, 10 ** width)
            m = hi - lo
            idx = np.arange(lo, hi, dtype=np.int64)
            rec = np.empty((m, 1 + len(lab) + width + len(suffix) + 1 + RL + 3 + RL + 1), np.uint8)
            rec[:, 0] = ord("@")
            c = 1
            rec[:, c:c + len(lab)] = np.frombuffer(lab, np.uint8)
            c += len(lab)
            for k in range(width):
                rec[:, c + k] = (idx // 10 ** (width - 1 - k)) % 10 + ord("0")
            c += width
            rec[:, c:c + len(suffix)] = np.frombuffer(suffix, np.uint8)
            c += len(suffix)
            rec[:, c] = 10
            c += 1
            rec[:, c:c + RL] = arr[lo * RL:hi * RL].reshape(m, RL)
            c += RL
            rec[:, c:c + 3] = np.frombuffer(b"\n+\n", np.uint8)
            c += 3
            rec[:, c:c + RL] = ord("I")
            c += RL
            rec[:, c] = 10
            f.write(rec.tobytes())
            lo = hi
            width += 1


def write_fastq_pair(prefix, r1, r2, n, RL, label="p", mode="wb"):
    write_fastq(prefix + "_1.fq", r1, n, RL, label, b"/1", mode)
    if r2 is not None:
        write_fastq(prefix + "_2.fq", r2, n, RL, label, b"/2", mode)


class ReferenceRunner:
    """The UNMODIFIED reference binary (oracle/_ref/urmap) on the host cores.  Index load and start-up are taken out as
    the wall of a run over 4 reads (measured once); the reference's own summary lines ("Seconds to load index",
    "Seconds in mapper": whole seconds, state1.cpp:617-626) are reported beside that figure."""

    def __init__(self, ufi_path, workdir, threads):
        from oracle import oracle_py as O
        self.bin = O.REF_BIN
        self.ufi = ufi_path
        self.workdir = workdir
        self.threads = threads
        self.t_load = None
        # torchrun exports OMP_NUM_THREADS=1 to its workers and the reference caps -threads at omp_get_max_threads()
        # (myutils.cpp:129-147): give the baseline every host thread explicitly
        self.env = dict(os.environ, OMP_STACKSIZE="64M", OMP_NUM_THREADS=str(threads))

    def available(self):
        return os.path.exists(self.bin)

    def cmd(self, prefix, paired, sam, tab=None):
        c = ["-map2", prefix + "_1.fq", "-reverse", prefix + "_2.fq"] if paired else ["-map", prefix + "_1.fq"]
        return [self.bin] + c + ["-ufi", self.ufi, "-samout", sam, "-threads", str(self.threads)] + (["-tabbedout", tab] if tab else [])

    def _run(self, c, what):
        # The reference has no error channel but its exit status, and its multi-threaded mapper occasionally dies with
        # SIGSEGV on this workload (seen on the GPU box with 16 threads, not reproducible per input): a crashed
        # attempt is logged and repeated.
        for attempt in range(4):
            t0 = time.time()
            p = subprocess.run(c, capture_output=True, env=self.env)
            if p.returncode == 0:
                return time.time() - t0, (p.stdout + p.stderr).decode(errors="replace")
            log(f"reference {what} run exited {p.returncode} (attempt {attempt + 1}): "
                f"{p.stderr.decode(errors='replace')[-200:]!r}")
        raise RuntimeError(f"reference {what} run failed {attempt + 1} times with exit status {p.returncode}")

    def load_seconds(self, prefix, paired):
        if self.t_load is None:
            tiny = os.path.join(self.workdir, "tiny")
            for sfx in ("_1.fq", "_2.fq"):
                if os.path.exists(prefix + sfx):
                    with open(prefix + sfx, "rb") as f, open(tiny + sfx, "wb") as g:
                        for _ in range(16):
                            g.write(f.readline())
            self.t_load, _ = self._run(self.cmd(tiny, paired, tiny + ".sam"), "index-load (4 reads)")
        return self.t_load

    def run(self, prefix, paired, n_reads, sam, what="sample", tab=None):
        t_load = self.load_seconds(prefix, paired)
        t_run, text = self._run(self.cmd(prefix, paired, sam, tab), what)
        dt = max(t_run - t_load, 1e-3)
        own = {}
        m = re.search(r"(\d+)\s+Seconds to load index", text)
        if m:
            own["seconds_to_load_index"] = int(m.group(1))
        m = re.search(r"([0-9.]+)\s+(Seconds|Minutes) in mapper", text)
        if m:
            own["seconds_in_mapper"] = float(m.group(1)) * (60.0 if m.group(2) == "Minutes" else 1.0)
        m = re.search(r"(\S+)\s+Reads/sec\. \((\d+) threads\)", text)
        if m:
            own["reads_per_sec_line"] = m.group(1)
            own["threads"] = int(m.group(2))
        return {"reads": n_reads, "seconds": dt, "wall_seconds": t_run, "load_seconds": t_load, "reads_per_s": n_reads / dt,
                "sam": sam, "reference_summary": own}


def samdiff(a, b, unmatched=None):
    exe = os.path.join(ROOT, "urmap_b200", "bin", "samdiff")
    p = subprocess.run([exe, a, b] + ([unmatched] if unmatched else []), capture_output=True, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"samdiff failed: {p.stderr[-200:]!r}")
    return json.loads(p.stdout)


def run_cli_once(prefix, paired, ufi_path, sam, threads, tab=None, **env):
    """`urmap_b200 -map/-map2 ... -samout [-tabbedout]` (FASTQ files in, SAM file out); returns its stage times."""
    exe = os.path.join(ROOT, "urmap_b200", "bin", "urmap_b200")
    c = ["-map2", prefix + "_1.fq", "-reverse", prefix + "_2.fq"] if paired else ["-map", prefix + "_1.fq"]
    t0 = time.time()
    p = subprocess.run([exe] + c + ["-ufi", ufi_path, "-samout", sam, "-threads", str(threads)] + (["-tabbedout", tab] if tab else []),
                       capture_output=True, env=dict(os.environ, URMB_PROFILE="1", **env))
    wall = time.time() - t0
    err = p.stderr.decode(errors="replace")
    if p.returncode != 0:
        raise RuntimeError(f"urmap_b200 exited {p.returncode}: {err[-300:]!r}")
    prof = [ln[len("[urmb host] "):] for ln in err.splitlines() if ln.startswith("[urmb host]")]
    m = re.search(r"load ([0-9.]+)s.*mapper total ([0-9.]+)s", " ".join(prof))
    if not m:
        raise RuntimeError("urmap_b200 printed no stage times")
    warn = [ln for ln in err.splitlines() if "WARNING" in ln]
    return {"wall_seconds": wall, "seconds_to_load_index": float(m.group(1)), "seconds_in_mapper": float(m.group(2)),
            "host_profile": prof, "warnings": warn}


def run_cli(ufi_path, prefix, cli_prefix, n_units, paired, threads, ref_sam):
    """The drop-in itself over n_units pairs whose first part is the sample the reference was timed on; value = reads /
    its own 'Seconds in mapper' (index load excluded the way the reference excludes it, state1.cpp:617-626); its SAM file
    is compared with the reference's record by record (tools/samdiff.cpp)."""
    reads = n_units * (2 if paired else 1)
    r = run_cli_once(cli_prefix, paired, ufi_path, cli_prefix + "_cli.sam", threads)
    out = {"value": reads / r["seconds_in_mapper"], "unit": "reads/s", "reads": reads, "host_threads": threads,
           "what": "urmap_b200 CLI, FASTQ files -> SAM file in /dev/shm; reads / its own 'Seconds in mapper' (first batch "
                   "read to SAM file closed)", **r}
    for key, sam, env in (("to_dev_null", "/dev/null", {}), ("write2", cli_prefix + "_cli2.sam", {"URMB_NO_MMAP_OUT": "1"})):
        try:
            r2 = run_cli_once(cli_prefix, paired, ufi_path, sam, threads, **env)
            out[key] = {"value": reads / r2["seconds_in_mapper"], "unit": "reads/s", **r2}
        except Exception as e:
            out[key] = {"error": repr(e)}
        if sam != "/dev/null" and os.path.exists(sam):
            os.unlink(sam)
    if ref_sam and os.path.exists(ref_sam):
        # the reference mapped the first part of the CLI's input: cut the CLI's SAM at that many records
        d = samdiff_prefix(ref_sam, cli_prefix + "_cli.sam")
        out["sam_vs_reference"] = d
    return out


def samdiff_prefix(ref_sam, cli_sam):
    """Identity of the reference's records with the same records of a CLI run over a superset of the reads: the CLI's
    file is cut after as many record lines as the reference's has (the CLI writes records in input order)."""
    n_ref = 0
    with open(ref_sam, "rb") as f:
        for ln in f:
            if not ln.startswith(b"@"):
                n_ref += 1
    cut = cli_sam + ".head"
    with open(cli_sam, "rb") as f, open(cut, "wb") as g:
        k = 0
        for ln in f:
            if ln.startswith(b"@"):
                g.write(ln)
                continue
            if k >= n_ref:
                break
            g.write(ln)
            k += 1
    d = samdiff(ref_sam, cut, os.environ.get("URMB_BENCH_UNMATCHED") and os.environ["URMB_BENCH_UNMATCHED"] + "_main.txt")
    os.unlink(cut)
    return {"records": d["records_a"], "identical": d["identical"], "header_equal": d["header_equal"], "pct": d["pct"],
            "cli_records_compared": d["records_b"]}


def run_port_cpu(ufi_path, a1, a2, n_units, RL, paired, threads):
    """Fallback baseline when the reference binary is unavailable or crashed: the CPU restatement (oracle port)."""
    from oracle import oracle_py as O
    o = (np.arange(n_units + 1, dtype=np.uint32) * RL)
    oix = O.Index(ufi_path)
    b1 = O.ReadBatch(np.ascontiguousarray(a1[:n_units * RL]), o)
    t0 = time.time()
    if paired:
        O.map_pe(oix, b1, O.ReadBatch(np.ascontiguousarray(a2[:n_units * RL]), o), threads=threads)
    else:
        O.map_se(oix, b1, threads=threads)
    dt = time.time() - t0
    oix.close()
    reads = n_units * (2 if paired else 1)
    return {"reads": reads, "seconds": dt, "load_seconds": 0.0, "reads_per_s": reads / dt, "sam": None}


def work_per_read(ufi_path, batch, n_units, RL, paired):
    """Work counters of the reference's control flow (oracle port) on a sample of this workload; B_algo = 5*P + 5*H + C
    (SURVEY.md §8d) split over the kernels that do the work."""
    from oracle import oracle_py as O
    _, _, a1, a2, offs = batch
    o = np.ascontiguousarray(offs[:n_units + 1])
    oix = O.Index(ufi_path)
    if paired:
        *_, st = O.map_pe(oix, O.ReadBatch(np.ascontiguousarray(a1[:n_units * RL]), o),
                          O.ReadBatch(np.ascontiguousarray(a2[:n_units * RL]), o), threads=os.cpu_count(), want_stats=True)
    else:
        *_, st = O.map_se(oix, O.ReadBatch(np.ascontiguousarray(a1[:n_units * RL]), o), threads=os.cpu_count(),
                          want_stats=True)
    oix.close()
    r = max(1, st["reads"])
    per = {k: st[k] / r for k in ("probes", "row_hops", "row_hops_long", "compare_bytes", "compare_bytes_rows",
                                  "compare_bytes_rows_long", "dp_cells", "dp_cells_scan", "dp_calls", "scan_calls",
                                  "extend_calls")}
    per["bytes"] = 5 * per["probes"] + 5 * per["row_hops"] + per["compare_bytes"]
    # attribution: slot probes + seed extensions (probe kernel) / list hops + row-candidate extensions of the first
    # visit (rows kernel) / of the second visit of rows longer than 2 (rows_long kernel)
    per["bytes_rows_long"] = 5 * per["row_hops_long"] + per["compare_bytes_rows_long"]
    per["bytes_rows"] = 5 * per["row_hops"] + per["compare_bytes_rows"] - per["bytes_rows_long"]
    per["bytes_probe"] = per["bytes"] - per["bytes_rows"] - per["bytes_rows_long"]
    return per


SURVEY_WORK = {"probes": 157.0, "row_hops": 50.0, "row_hops_long": 25.0, "compare_bytes": 2213.0, "compare_bytes_rows": 1100.0,
               "compare_bytes_rows_long": 500.0, "dp_cells": 669.0, "dp_cells_scan": 150.0,
               "bytes": 5 * 157 + 5 * 50 + 2213.0, "bytes_rows": 5 * 25 + 600.0, "bytes_rows_long": 5 * 25 + 500.0,
               "bytes_probe": 5 * 157 + 1113.0, "source": "SURVEY.md §8d constants (split over the row kernels estimated)"}

# kernel class -> (kernel name(s), kind); kind "gather": HBM random gathers, "dp": dynamic programming, "state": replay of
# the order-dependent bookkeeping over data the gather kernels produced
KCLASS = {
    "probe": ("probe_pair_kernel | probe_kernel", "gather"), "pair": ("pair_kernel | seed_kernel_se", "state"),
    "align_a": ("align_kernel_a | align_kernel_se3", "dp"), "rows": ("rows_kernel | rows_kernel_se", "gather"),
    "rows_long": ("rows_long_kernel | rows_long_kernel_se", "gather"), "align_c": ("align_kernel_c | align_kernel_se6", "dp"),
    "finish": ("finish_kernel", "state"), "rescue": ("rescue_scan_kernel", "gather"), "rescue_last": ("rescue_last_kernel", "dp"),
    "rescue_dp": ("rescue_dp_kernel", "dp"),
    "rescue_legacy": ("rescue_kernel", "state"),
}


NSLOTS = int(os.environ.get("URMB_BENCH_SLOTS", "6"))   # batch slots the bench keeps in flight (the context has 8): the side-stream work of a batch -- mate rescue,
             # big-capacity rerun of the few reads over a capacity, occasionally 100+ ms for one heavy pair -- then has
             # five steps to finish before its slot is needed again


def time_steps(ctx, batches, paired, steps, warmup, D, device, keep_last=False):
    """K steps issued back to back with the inputs resident in HBM: device time between two context-wide CUDA events,
    per-kernel-class launch durations (CUDA events around every launch) of the last steps.  keep_last: also return
    copies of the results of step K-1 (r1, r2, runs) as `last`."""
    import torch
    nb = len(batches)
    B = len(batches[0][4]) - 1
    for w in range(max(warmup, 3)):   # warm-up (also sizes the slots' buffers)
        _, _, a1, a2, offs = batches[w % nb]
        ctx.submit(w % NSLOTS, a1, offs, a2, offs if paired else None)
        ctx.wait(w % NSLOTS, B, paired)
    for s in range(NSLOTS):
        _, _, a1, a2, offs = batches[s % nb]
        ctx.upload(s, a1, offs, a2, offs if paired else None)
    D.barrier()
    torch.cuda.synchronize()
    launches0 = ctx.launch_count()
    t_wall0 = time.perf_counter()
    # the mate-rescue kernels of step k run on a side stream and overlap step k+1; the end mark waits for the last ones
    ctx.mark(0)
    for k in range(steps):
        ctx.launch(k % NSLOTS)
    ctx.mark(1)
    dev_ms = ctx.mark_elapsed()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    gpu_launches = ctx.launch_count() - launches0
    nlast = min(3, steps)
    kms, klaunch = {}, {}
    for k in range(steps - nlast, steps):
        tm = ctx.timing(k % NSLOTS)
        for name, v in tm["kernel_ms"].items():
            if tm["kernel_launches"][name]:
                kms[name] = kms.get(name, 0.0) + v / nlast
                klaunch[name] = klaunch.get(name, 0) + tm["kernel_launches"][name]
    klaunch = {k: max(1, v // nlast) for k, v in klaunch.items()}
    last = None
    for s in range(min(NSLOTS, steps)):   # drain
        ctx.download(s)
        r1, r2, runs = ctx.wait(s, B, paired)
        if keep_last and s == (steps - 1) % NSLOTS:
            last = (r1.copy(), None if r2 is None else r2.copy(), runs.copy())
    # pairs the probe kernel's first look finished (seed-loop exit of Search4/5) in the last batch of slot 0
    first_look = ctx.first_look_count(0)[0] / float(B) if paired else 0.0
    return {"dev_ms": dev_ms, "wall_ms": 1e3 * t_wall, "gpu_launches": gpu_launches, "kernel_ms": kms, "kernel_launches": klaunch,
            "first_look_frac": first_look, "last": last}


DUMP_SAMPLE = 100_000   # reads per mate: 4 MB of result fields per mate, plus the path runs of those reads


def dump_outputs(out_dir, last, seed=0):
    """The results of one step as .npy files: for a fixed, seeded sample of the batch's reads (`sample_index`), every
    result field per mate (`mate1_<field>`, `mate2_<field>` when paired; db_pos in float64, the rest in float32) and the
    path runs of the sampled reads in sample order (`mateN_path`, `mateN_path_runs` long each).  The pool offsets of the
    paths are left out: they depend on the order in which warps finish."""
    r1, r2, runs = last
    n = len(r1)
    idx = np.sort(np.random.default_rng(seed).choice(n, size=min(n, DUMP_SAMPLE), replace=False))
    arrays = {"sample_index": idx.astype(np.float64)}
    for m, r in ((1, r1), (2, r2)):
        if r is None:
            continue
        s = r[idx]
        for f in ("db_pos", "score", "best", "second", "mapq", "flags", "hit_count", "hsp_count", "path_runs"):
            arrays[f"mate{m}_{f}"] = s[f].astype(np.float64 if f == "db_pos" else np.float32)
        lens = s["path_runs"].astype(np.int64)
        starts = np.repeat(s["path_off"].astype(np.int64), lens)
        within = np.arange(int(lens.sum())) - np.repeat(np.cumsum(lens) - lens, lens)
        arrays[f"mate{m}_path"] = runs[starts + within].astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise RuntimeError(f"--dump-outputs: {total} bytes, over the 64 MB bound")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "arrays": len(arrays), "bytes": total}


def time_e2e(ctx, batches, paired, steps, D, device):
    """Host buffers in, host buffers out through the C ABI, NSLOTS slots in flight."""
    import torch
    nb = len(batches)
    B = len(batches[0][4]) - 1
    D.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d2h = 0
    trace = [] if os.environ.get("URMB_E2E_TRACE") else None   # host seconds spent in every wait / submit call
    for k in range(steps):
        if k >= NSLOTS:
            ta = time.perf_counter()
            r1, r2, runs = ctx.wait(k % NSLOTS, B, paired)
            if trace is not None:
                trace.append(("wait", k - NSLOTS, time.perf_counter() - ta))
            d2h += r1.nbytes + (r2.nbytes if r2 is not None else 0) + runs.nbytes + 16
        _, _, a1, a2, offs = batches[k % nb]
        ta = time.perf_counter()
        ctx.submit(k % NSLOTS, a1, offs, a2, offs if paired else None)
        if trace is not None:
            trace.append(("submit", k, time.perf_counter() - ta))
    for k in range(max(0, steps - NSLOTS), steps):
        ta = time.perf_counter()
        r1, r2, runs = ctx.wait(k % NSLOTS, B, paired)
        if trace is not None:
            trace.append(("wait", k, time.perf_counter() - ta))
        d2h += r1.nbytes + (r2.nbytes if r2 is not None else 0) + runs.nbytes + 16
    torch.cuda.synchronize()
    t1 = time.perf_counter() - t0
    if trace is not None:
        log("e2e trace (ms): " + " ".join(f"{w}{k}={1e3 * t:.1f}" for w, k, t in trace))
        tm = ctx.timing((steps - 1) % NSLOTS)
        log(f"e2e last batch: h2d {tm['h2d_ms']:.2f} ms, d2h {tm['d2h_ms']:.2f} ms (copy engine time of one batch)")
    return t1, d2h


def rooflines(kms, klaunch, algo, reads_per_step, rpu, RL, W, peaks, micro, traffic, first_look=0.0):
    """One object per kernel class that ran: share of the step, average launch duration, and the roofline that bounds it
    (HBM bytes for the gather kernels, int32 ALU ops for the DP kernels)."""
    peak = peaks.get("hbm_gbs")
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peak else "fallback 6650 GB/s (B200_PROFILING.md)"
    peak = peak or 6650.0
    qwc = max(1, RL - W + 1)
    total = max(sum(kms.values()), 1e-9)
    dp_flank = max(algo.get("dp_cells", 0.0) - algo.get("dp_cells_scan", 0.0), 0.0)
    # algorithmic bytes per read by class (SURVEY.md §8d: B_algo = 5 P + 5 H + C of the reference's control flow)
    byts = {
        "probe": (algo["bytes_probe"], "5 B x slot probes + compared bases of BOTH1 seed extensions (reference control flow)"),
        "rows": (algo["bytes_rows"], "5 B x list hops + compared bases of row-candidate extensions, first visit (rows <= 2 extended)"),
        "rows_long": (algo["bytes_rows_long"], "5 B x list hops + compared bases of the deferred rows longer than 2"),
        "pair": (2 * qwc * 9 + 384.0, "its inputs read once: probe rows (tally, pos, packed extension: 9 B x 2 strands x k-mers) + staged read"),
        "align_a": (0.5 * dp_flank / 25.0 + RL, "genome windows of the flank DPs (cells / band width) + the read; DP kernel: see roofline_dp_alu"),
        "align_c": (0.5 * dp_flank / 25.0 + RL, "genome windows of the flank DPs (cells / band width) + the read; DP kernel: see roofline_dp_alu"),
        "rescue": (algo.get("scan_calls", 0.0) * 1100.0, "scanned window bytes (1024 + 2 QL per scan)"),
        "rescue_dp": (algo.get("dp_cells_scan", 0.0) / max(RL, 1), "window bytes of the full-window DPs; DP kernel: see roofline_dp_alu"),
        # the in-place mate rescue (URMB_RESCUE_ROUNDS=0, the default): window scans and full-window DPs in one kernel
        "rescue_last": (algo.get("scan_calls", 0.0) * 1100.0 + algo.get("dp_cells_scan", 0.0) / max(RL, 1),
                        "scanned window bytes (1024 + 2 QL per scan) + window bytes of the full-window DPs (run in place by the pair's warp)"),
    }
    out = {}
    for cls, ms in kms.items():
        name, kind = KCLASS.get(cls, (cls, "state"))
        launches = klaunch.get(cls, 1)
        avg_s = ms / 1e3 / launches
        o = {"kernel": name, "kind": kind, "ms_per_step": ms, "share_of_step": ms / total, "launches_per_step": launches,
             "avg_launch_ms": 1e3 * avg_s}
        if cls in byts:
            b, what = byts[cls]
            ach = b * (reads_per_step / launches) / max(avg_s, 1e-9) / 1e9
            tr = traffic.get(name.split(" | ")[0])
            o.update({"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                      "traffic": (tr["dram_bytes_per_pair"] * (reads_per_step / launches / rpu)) if tr else None,
                      "peak_source": peak_src, "algorithmic_bytes_per_read": b, "algorithmic_bytes": what})
        out[cls] = o
    roof_gather, roof_alu = None, None
    if micro:
        # slot probes the kernel makes per read: every k-mer of both strands, except for the pairs its first look finishes
        # (16 probes per read there, which the other pairs make on top)
        apr = 2.0 * qwc * (1.0 - first_look) + (16.0 if rpu == 2 and first_look > 0 else 0.0)
        acc = apr * reads_per_step / max(kms.get("probe", 0.0) / 1e3, 1e-9) / 1e9
        pk = micro["gather_4B"]["gaccess_per_s"]
        roof_gather = {"kernel": "probe_pair_kernel | probe_kernel", "bound": "hbm random sector gather", "achieved": acc, "peak": pk,
                       "unit": "G accesses/s", "frac": acc / pk, "accesses_per_read": apr,
                       "peak_source": "urmb_peak_gather: random 4-byte reads at 32-byte-aligned addresses over the blob",
                       "peak_16B_gaccess_per_s": micro["gather_16B"]["gaccess_per_s"]}
        dp_classes = [c for c in ("align_a", "align_c", "rescue_dp") if c in kms and kms[c] > 0]
        cells = algo.get("dp_cells", 0.0) * reads_per_step
        if "rescue_dp" not in dp_classes:
            # the full-window DPs of the mate rescue run inside the in-place rescue kernel, whose time is mostly window scans:
            # their cells are left out and the figure is that of the flank DPs alone
            cells -= algo.get("dp_cells_scan", 0.0) * reads_per_step
        align_ms = sum(kms[c] for c in dp_classes)
        if cells and align_ms > 0:
            ach = 16.0 * cells / (align_ms / 1e3) / 1e12
            roof_alu = {"kernels": " + ".join(KCLASS[c][0] for c in dp_classes),
                        "cells": "flank DPs and batched rescue DPs" if "rescue_dp" in dp_classes else "flank DPs (rescue DPs run in place in rescue_last_kernel: not counted)",
                        "bound": "int32 alu",
                        "achieved": ach, "peak": micro["alu"]["tops_per_s"], "unit": "Tops/s",
                        "frac": ach / micro["alu"]["tops_per_s"], "dp_cells_per_s": cells / (align_ms / 1e3),
                        "ops_per_cell": 16, "kernel_ms": align_ms,
                        "peak_source": "urmb_peak_alu: independent LOP3/IADD chains on all SMs"}
    return out, roof_gather, roof_alu


def main():
    # the contract is ONE JSON line on stdout: libraries that write to fd 1 (NCCL prints its version there) get stderr
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="urmb", choices=["urmb", "reference"])
    ap.add_argument("--genome-len", type=int, default=3_100_000_000)
    ap.add_argument("--segdup-frac", type=float, default=0.03)
    ap.add_argument("--tandem-frac", type=float, default=0.01)
    ap.add_argument("--pairs-per-step", type=int, default=1_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--sub", type=float, default=0.01)
    ap.add_argument("--indel", type=float, default=0.001)
    ap.add_argument("--single-end", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE.json configurations")
    ap.add_argument("--only-configs", default="", help="comma-separated keys of EXTRA_CONFIGS to run (default: all)")
    ap.add_argument("--config-steps", type=int, default=5)
    ap.add_argument("--config-units-scale", type=float, default=1.0)
    ap.add_argument("--cpu-sample-pairs", type=int, default=1_000_000)
    ap.add_argument("--ref-min-seconds", type=float, default=32.0, help="--impl reference: seconds the mapper must run")
    ap.add_argument("--workdir", default=os.environ.get("URMB_BENCH_DIR"),
                    help="scratch files (UFI, FASTQ, SAM); default: a new private directory under /dev/shm")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (a fixed sample of its reads) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    paired = not args.single_end
    rpu = 2 if paired else 1

    import torch

    from urmap_b200 import dist as D
    rank, local_rank, world = D.env_rank()
    if args.impl == "reference" and rank != 0:
        return 0
    if args.impl == "urmb":
        D.init()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the mapping engine has no CPU path")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    from urmap_b200 import engine
    from urmap_b200 import build as BLD
    if not BLD.is_current():   # asks make without building: the tree may be read-only here
        raise SystemExit("liburmb.so or the CLI is older than its sources: run __graft_entry__.build() first")
    engine.lib()

    baseline = load_json("BASELINE.json")
    peaks = load_json("MEASURED_PEAKS.json")
    metric = baseline.get("metric", "reads/s mapped, 2x150bp human-scale")
    human = args.genome_len >= 100_000_000
    meta, seq, blob = build_workload(args, rank, world if args.impl == "urmb" else 1, device)
    workload = ("synthetic %.2f Gb reference (%d contigs, 10%% interspersed repeats, %.0f%% segmental duplications, %.0f%% "
                "tandem repeats), UFI in HBM, %s%d bp reads, %.1f%% subs + %.2f%% indels"
                % (args.genome_len / 1e9, 24 if human else 3, 100 * meta.get("segdup_frac", 0), 100 * meta.get("tandem_frac", 0),
                   "paired-end 2x" if paired else "single-end ", args.read_len, 100 * args.sub, 100 * args.indel))
    cfg = {"workload": workload, "baseline_config": 2 if paired else 1,
           "pairs_per_step_per_gpu" if paired else "reads_per_step_per_gpu": args.pairs_per_step,
           "parallelism": f"reads sharded over {world} GPU(s), index replicated by NCCL broadcast, no per-batch collective",
           "slots_in_flight": NSLOTS,
           "l2_policy": "inputs larger than L2: each batch is >=300 MB of reads and probes a 27 GB table at random",
           "pe_method": 4, "method": 6}
    nb = 3
    B, RL = args.pairs_per_step, args.read_len
    batches = make_batches(meta, seq, device, nb, B, paired, RL, args.sub, args.indel, seed0=1000 * (rank + 1))
    own_workdir = args.workdir is None
    if own_workdir:
        args.workdir = tempfile.mkdtemp(prefix="urmb_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    else:
        os.makedirs(args.workdir, exist_ok=True)
    # scratch files reach tens of GB at human scale (the UFI file) and /dev/shm is RAM: removed however the run ends
    if (own_workdir or args.workdir.startswith("/dev/shm")) and (own_workdir or rank == 0) \
            and not os.environ.get("URMB_KEEP_BENCH_DIR"):
        atexit.register(shutil.rmtree, args.workdir, True)
    ufi_path = os.path.join(args.workdir, "bench.ufi")
    prefix = os.path.join(args.workdir, "sample")
    threads = os.cpu_count()

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        t0 = time.time()
        write_ufi_file(ufi_path, meta, seq, blob)
        log(f"UFI file written for the reference in {time.time() - t0:.1f}s")
        a1 = np.concatenate([b[2] for b in batches])
        a2 = None if not paired else np.concatenate([b[3] for b in batches])
        n_dist = B * nb
        write_fastq_pair(prefix, a1, a2, n_dist, RL)
        del seq, blob
        torch.cuda.empty_cache()
        ref = ReferenceRunner(ufi_path, args.workdir, threads)
        kind, r, sample = "reference", None, None
        if ref.available():
            try:
                # pass 1: the distinct reads once.  BASELINE.md §3: a run under 30 s in the mapper is repeated with
                # more reads -- the same files concatenated as often as the first pass says is needed
                r = ref.run(prefix, paired, n_dist * rpu, "/dev/null", "sample (pass 1)")
                reps = 1
                if r["seconds"] < args.ref_min_seconds:
                    reps = int(np.ceil(1.1 * args.ref_min_seconds / r["seconds"]))
                    big = os.path.join(args.workdir, "sample_rep")
                    for sfx in ("_1.fq", "_2.fq"):
                        if os.path.exists(prefix + sfx):
                            with open(big + sfx, "wb") as g:
                                for _ in range(reps):
                                    with open(prefix + sfx, "rb") as f:
                                        shutil.copyfileobj(f, g, 1 << 24)
                    first = r
                    r = ref.run(big, paired, n_dist * rpu * reps, "/dev/null", f"sample x{reps}")
                    r["first_pass"] = {k: first[k] for k in ("reads", "seconds", "reads_per_s", "reference_summary")}
                sample = (f"{n_dist} distinct {'pairs' if paired else 'reads'} of the workload x {reps} (one urmap process, "
                          f"-threads {threads}, SAM to /dev/null): {r['reads']} reads in {r['seconds']:.1f}s = wall "
                          f"{r['wall_seconds']:.1f}s minus the wall of a 4-read run (index load {r['load_seconds']:.1f}s); "
                          f"the reference's own summary: {r['reference_summary']}")
            except RuntimeError as e:
                log(f"WARNING: {e}")
                r = None
        if r is None:
            # LOUD: a port number is not the reference's; the driver's ratio against it is void
            log("WARNING: the reference binary is unavailable or crashed; this line times the CPU RESTATEMENT "
                "(oracle port) instead -- kind 'port', any ratio against it is VOID")
            kind = "port"
            n_port = min(n_dist, 200_000)
            r = run_port_cpu(ufi_path, a1, a2, n_port, RL, paired, threads)
            r["reference_summary"] = {}
            sample = (f"{n_port} {'pairs' if paired else 'reads'} of the same workload through the CPU restatement "
                      f"(oracle/urmap_oracle.cpp, OpenMP over reads; REFERENCE BINARY UNAVAILABLE: ratio void)")
        per_step = r["reads"] // rpu // args.steps
        cfg_ref = dict(cfg)
        cfg_ref["pairs_per_step_per_gpu" if paired else "reads_per_step_per_gpu"] = per_step
        cfg_ref["note"] = (f"{args.steps} steps x {per_step} {'pairs' if paired else 'reads'}: a bounded sample of the "
                           f"workload per step, one process over all of them")
        line = {"impl": "reference", "metric": metric, "value": r["reads_per_s"], "unit": "reads/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32/fp32",
                "data": "synthetic", "config": cfg_ref,
                "cpu_baseline": {"value": r["reads_per_s"], "unit": "reads/s", "cores": threads, "kind": kind,
                                 "sample": sample},
                "e2e": {"value": r["reads_per_s"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "reference_summary": r.get("reference_summary"), "seconds_in_mapper_wall_minus_load": r["seconds"],
                "first_pass": r.get("first_pass"), "ratio_void": kind != "reference",
                "index_built_by": "urmb_build_index_device on the GPU (byte-identical UFI; setup, not timed)",
                "load_seconds": r["load_seconds"]}
        print(json.dumps(line), file=_OUT, flush=True)
        return 0

    # ------------------------------------------------------------------ urmb arm
    ctx = engine.Context(local_rank)
    ctx.attach_index(meta["word_length"], meta["max_ix"], meta["seq_data_size"], meta["slot_count"], blob.data_ptr(),
                     seq.data_ptr(), keepalive=(seq, blob))

    # measured denominators of the two rooflines (SURVEY.md §8d): random sector gathers over the 27 GB blob, int32 ALU rate
    micro = None
    if rank == 0:
        try:
            torch.cuda.synchronize()
            micro = {"gather_4B": engine.peak_gather(blob.data_ptr(), 5 * meta["slot_count"] // 32 * 32, 4),
                     "gather_16B": engine.peak_gather(blob.data_ptr(), 5 * meta["slot_count"] // 32 * 32, 16),
                     "alu": engine.peak_alu()}
            log(f"micro-benchmarks: {micro}")
        except Exception as e:
            log(f"micro-benchmarks failed: {e!r}")
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.active = True
    # ---- value: inputs resident in HBM, kernels only, CUDA events on the launching stream
    tv = time_steps(ctx, batches, paired, args.steps, args.warmup, D, device, keep_last=bool(args.dump_outputs))
    sampler.active = False
    if args.dump_outputs and rank == 0:
        log(f"outputs of the last timed step: {dump_outputs(args.dump_outputs, tv.pop('last'))}")
    D.barrier()
    kms, klaunch = tv["kernel_ms"], tv["kernel_launches"]
    dev_ms_max = D.max_over_ranks(tv["dev_ms"], device)
    total_reads = rpu * B * args.steps * world
    value = total_reads / (dev_ms_max / 1e3)
    # ---- e2e: host buffers in, host buffers out, three slots in flight
    sampler.active = True
    t_e2e, d2h = time_e2e(ctx, batches, paired, args.steps, D, device)
    sampler.active = False
    D.barrier()
    t_e2e_max = D.max_over_ranks(t_e2e, device)
    e2e_value = total_reads / t_e2e_max
    h2d_per_step = rpu * B * RL + 4 * (rpu * B + 1)
    clocks = sampler.summary()
    sampler.stop()
    log(f"main workload: {value / 1e6:.2f} M reads/s kernels, {e2e_value / 1e6:.2f} M e2e; kernel ms/step "
        + " ".join(f"{k}={v:.2f}" for k, v in kms.items()))

    # ---- the other BASELINE.json configurations (rank 0, N == 1 only): kernels timed the same way
    configs = {}
    cfg_batches = {}
    do_extra = rank == 0 and world == 1 and not args.no_configs
    if do_extra:
        only = [k for k in args.only_configs.split(",") if k]
        for ci, ec in enumerate(EXTRA_CONFIGS):
            if only and ec["key"] not in only:
                continue
            try:
                units = max(1000, int(ec["units"] * args.config_units_scale))
                t0 = time.time()
                bt = make_batches(meta, seq, device, 2, units, ec["paired"], ec["read_len"], ec["sub"], ec["indel"],
                                  seed0=50_000 + 100 * ci, enrich=ec["enrich"])
                t = time_steps(ctx, bt, ec["paired"], args.config_steps, 3, D, device)
                r_ = 2 if ec["paired"] else 1
                te, _ = time_e2e(ctx, bt, ec["paired"], args.config_steps, D, device)
                configs[ec["key"]] = {
                    "baseline_config": ec["baseline_config"], "workload": ec["what"],
                    "reads_per_step": r_ * units, "steps": args.config_steps,
                    "value": r_ * units * args.config_steps / (t["dev_ms"] / 1e3), "unit": "reads/s",
                    "ms_per_step": t["dev_ms"] / args.config_steps,
                    "e2e": {"value": r_ * units * args.config_steps / te, "unit": "reads/s"},
                    "kernel_ms_per_step": t["kernel_ms"], "kernel_launches_per_step": t["kernel_launches"],
                    "first_look_frac": t["first_look_frac"]}
                cfg_batches[ec["key"]] = bt[0]
                log(f"config {ec['key']}: {configs[ec['key']]['value'] / 1e6:.2f} M reads/s kernels "
                    f"({t['dev_ms'] / args.config_steps:.1f} ms per {r_ * units} reads; set-up {time.time() - t0:.1f}s); "
                    + " ".join(f"{k}={v:.2f}" for k, v in t["kernel_ms"].items()))
                del bt
            except Exception as e:
                configs[ec["key"]] = {"error": repr(e)}
                log(f"config {ec['key']} failed: {e!r}")

    # ---- cpu baseline, SAM identity and algorithmic bytes (rank 0, N == 1 only)
    cpu_baseline, sam_id, algo, cli = None, None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            t0 = time.time()
            write_ufi_file(ufi_path, meta, seq, blob)
            log(f"UFI file for the CPU baseline written in {time.time() - t0:.1f}s")
            n_cpu = min(args.cpu_sample_pairs, B)
            write_fastq_pair(prefix, batches[0][2], batches[0][3], n_cpu, RL)
            ref = ReferenceRunner(ufi_path, args.workdir, threads)
            r = None
            if ref.available():
                try:
                    r = ref.run(prefix, paired, n_cpu * rpu, prefix + "_ref.sam")
                except RuntimeError as e:
                    log(f"WARNING: {e}; cpu_baseline falls back to the oracle port (kind 'port')")
            if r is None:
                n_port = min(n_cpu, 200_000)
                rp = run_port_cpu(ufi_path, batches[0][2], batches[0][3], n_port, RL, paired, threads)
                cpu_baseline = {"value": rp["reads_per_s"], "unit": "reads/s", "cores": threads, "kind": "port",
                                "sample": f"first {n_port} {'pairs' if paired else 'reads'} of batch 0 through the CPU "
                                          f"restatement (oracle/urmap_oracle.cpp, OpenMP over reads)"}
            else:
                cpu_baseline = {"value": r["reads_per_s"], "unit": "reads/s", "cores": threads, "kind": "reference",
                                "sample": f"first {n_cpu} {'pairs' if paired else 'reads'} of batch 0; wall of "
                                          f"`urmap {'-map2' if paired else '-map'} -threads {threads}` minus the wall of a "
                                          f"4-read run (index load {r['load_seconds']:.1f}s excluded)",
                                "reference_summary": r["reference_summary"]}
                try:
                    n_cli = B * nb
                    write_fastq_pair(prefix + "_all", np.concatenate([b[2] for b in batches]),
                                     None if not paired else np.concatenate([b[3] for b in batches]), n_cli, RL)
                    cli = run_cli(ufi_path, prefix, prefix + "_all", n_cli, paired, threads, r["sam"])
                    for f in (prefix + "_all_1.fq", prefix + "_all_2.fq", prefix + "_all_cli.sam"):   # /dev/shm is finite
                        if os.path.exists(f):
                            os.unlink(f)
                    sam_id = cli.get("sam_vs_reference")
                    if sam_id:
                        sam_id = dict(sam_id, formatter="urmap_b200 CLI (SAM file of the drop-in against the SAM file of "
                                                        "the reference binary, tools/samdiff.cpp)")
                except Exception as e:
                    log(f"cli leg failed: {e!r}")
                # the other configurations: one reference run and one run of the drop-in per kind (single-end / paired)
                # over the concatenated samples; records are told apart by their label prefix
                for kind_paired in (False, True):
                    keys = [ec["key"] for ec in EXTRA_CONFIGS if ec["paired"] == kind_paired and ec["key"] in cfg_batches]
                    if not keys:
                        continue
                    try:
                        px = os.path.join(args.workdir, "cfg_pe" if kind_paired else "cfg_se")
                        n_reads = 0
                        for i, key in enumerate(keys):
                            ec = next(e for e in EXTRA_CONFIGS if e["key"] == key)
                            _, _, a1, a2, offs = cfg_batches[key]
                            nu = len(offs) - 1
                            write_fastq_pair(px, a1, a2, nu, ec["read_len"], label=key + ".", mode="wb" if i == 0 else "ab")
                            n_reads += nu * (2 if kind_paired else 1)
                        # paired: the -tabbedout files (second pairs of FindPairs, outputtab2.cpp:85-119) are compared as well
                        rtab, ctab = (px + "_ref.tab", px + "_cli.tab") if kind_paired else (None, None)
                        rr = ref.run(px, kind_paired, n_reads, px + "_ref.sam", "configs " + ",".join(keys), tab=rtab)
                        rc = run_cli_once(px, kind_paired, ufi_path, px + "_cli.sam", threads, tab=ctab)
                        d = samdiff(px + "_ref.sam", px + "_cli.sam", os.environ.get("URMB_BENCH_UNMATCHED") and
                                    os.environ["URMB_BENCH_UNMATCHED"] + ("_pe" if kind_paired else "_se") + ".txt")
                        dt_ = samdiff(rtab, ctab, os.environ.get("URMB_BENCH_UNMATCHED") and
                                      os.environ["URMB_BENCH_UNMATCHED"] + "_pe_tab.txt") if kind_paired else None
                        for key in keys:
                            g = d["groups"].get(key, {})
                            configs[key]["sam_identity"] = {"records": g.get("records_a", 0), "identical": g.get("identical", 0),
                                                            "pct": g.get("pct", 0.0), "cli_records": g.get("records_b", 0),
                                                            "header_equal": d["header_equal"]}
                            if dt_:
                                gt = dt_["groups"].get(key, {})
                                configs[key]["tabbedout_identity"] = {"lines": gt.get("records_a", 0), "identical": gt.get("identical", 0),
                                                                      "pct": gt.get("pct", 0.0), "cli_lines": gt.get("records_b", 0)}
                        for key in keys:
                            configs[key]["combined_run"] = {
                                "configs": keys, "reads": n_reads,
                                "reference_reads_per_s": rr["reads_per_s"], "reference_seconds": rr["seconds"],
                                "reference_summary": rr["reference_summary"],
                                "cli_reads_per_s": n_reads / rc["seconds_in_mapper"], "cli_seconds_in_mapper": rc["seconds_in_mapper"],
                                "cli_warnings": rc["warnings"]}
                        log(f"configs {keys}: SAM identity {[configs[k]['sam_identity']['pct'] for k in keys]}; reference "
                            f"{rr['reads_per_s'] / 1e6:.3f} M reads/s, CLI {n_reads / rc['seconds_in_mapper'] / 1e6:.2f} M reads/s")
                        if dt_:
                            log(f"configs {keys}: -tabbedout identity {[configs[k]['tabbedout_identity']['pct'] for k in keys]}")
                        for sfx in ("_1.fq", "_2.fq", "_ref.sam", "_cli.sam", "_ref.tab", "_cli.tab"):
                            if os.path.exists(px + sfx):
                                os.unlink(px + sfx)
                    except Exception as e:
                        log(f"identity leg of configs {keys} failed: {e!r}")
                        for key in keys:
                            configs[key]["sam_identity"] = {"error": repr(e)}
            algo = work_per_read(ufi_path, batches[0], min(50_000, B), RL, paired)
            for key, bt in cfg_batches.items():
                ec = next(e for e in EXTRA_CONFIGS if e["key"] == key)
                try:
                    configs[key]["work_per_read"] = work_per_read(ufi_path, bt, min(20_000, len(bt[4]) - 1), ec["read_len"],
                                                                  ec["paired"])
                except Exception as e:
                    configs[key]["work_per_read"] = {"error": repr(e)}
        except Exception as e:  # the baseline is reported, never required
            log(f"cpu baseline failed: {e!r}")
    if algo is None:
        algo = dict(SURVEY_WORK)

    if rank == 0:
        reads_per_step = rpu * B
        traffic = load_json(os.path.join("profiles", "ncu_traffic.json"))   # dram bytes per pair from ncu --set full
        W = meta["word_length"]
        per_kernel, roof_gather, roof_alu = rooflines(kms, klaunch, algo, reads_per_step, rpu, RL, W, peaks, micro, traffic,
                                                      tv["first_look_frac"])
        # `roofline` = the largest kernel class on the step's critical path (the kernels of the compute stream, whose durations
        # add up to the step); the mate-rescue classes run beside the following batches on the slots' side streams -- their
        # launch durations are those of kernels waiting for room on busy SMs -- and the largest of them is reported as
        # `roofline_side_stream`.  `per_kernel` has every class.
        SIDE = ("rescue", "rescue_dp", "rescue_last", "rescue_legacy")
        main_classes = [c for c in per_kernel if c not in SIDE] or list(per_kernel)
        dominant = max(main_classes, key=lambda c: per_kernel[c]["ms_per_step"])
        side_classes = [c for c in per_kernel if c in SIDE and "frac" in per_kernel[c]]
        side_dom = max(side_classes, key=lambda c: per_kernel[c]["ms_per_step"]) if side_classes else None
        for key, c in configs.items():
            if "kernel_ms_per_step" in c:
                ec = next(e for e in EXTRA_CONFIGS if e["key"] == key)
                a = c.get("work_per_read")
                a = a if isinstance(a, dict) and "bytes" in a else dict(SURVEY_WORK)
                pk, _, ra = rooflines(c["kernel_ms_per_step"], c["kernel_launches_per_step"], a, c["reads_per_step"],
                                      2 if ec["paired"] else 1, ec["read_len"], W, peaks, micro, {})
                dom = max([k for k in pk if k not in SIDE] or list(pk), key=lambda k: pk[k]["ms_per_step"])
                c["roofline"] = dict(pk[dom], kernel_class=dom)
                c["roofline_dp_alu"] = ra
        line = {
            "metric": metric, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32 (fp32 DP cells, fp64 MAPQ)", "data": "synthetic",
            "config": cfg,
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": h2d_per_step,
                    "d2h_bytes_per_step": d2h // max(1, args.steps), "ms_per_step": 1e3 * t_e2e_max / args.steps},
            "gpu_launches": tv["gpu_launches"],
            "first_look_frac": tv["first_look_frac"],   # pairs finished by the probe kernel's first look (seed-loop exit, search2m4.cpp:79-142)
            "clocks": clocks,
            "roofline": dict(per_kernel[dominant], kernel_class=dominant),
            "roofline_side_stream": dict(per_kernel[side_dom], kernel_class=side_dom) if side_dom else None,
            "roofline_probe": per_kernel.get("probe"),
            "roofline_probe_gather": roof_gather,
            "roofline_dp_alu": roof_alu,
            "per_kernel": per_kernel,
            "micro": micro,
            "kernel_ms_per_step": dict(kms, wall_incl_launch_gaps=tv["wall_ms"] / args.steps,
                                       note="summed launch durations per kernel class; the rescue kernels overlap the next step"),
            "cpu_baseline": cpu_baseline,
            "sam_identity_vs_reference": sam_id,
            "configs": configs,
            "cli": cli,
            "work_per_read": algo,
            "index": {"slot_count": meta["slot_count"], "seq_data_size": meta["seq_data_size"],
                      "gpu_build_seconds": meta.get("build_seconds"), "indexed_positions": meta.get("indexed")},
        }
        print(json.dumps(line), file=_OUT, flush=True)
    ctx.close()
    D.finalize()
    return 0


if __name__ == "__main__":
    sys.exit(main())
