"""Start-up from a FASTA file (-ref) against start-up from a UFI file (-ufi) at BASELINE.json's full size: the 3.1 Gb synthetic
reference of bench.py is written as FASTA (as tools/index_scale.py does), its UFI file by `-make_ufi -gpu_build`, and the same
1 M pairs of 2x150 bp reads are mapped with `-ufi` and with `-ref`.  Reports the time to index-ready of each, the parse
kernels' time and rate, the build time, the peak device memory (nvidia-smi, sampled every 50 ms), the same with -gpus 8 when
eight GPUs are there, and the SAM identity of the two runs (bin/samdiff).  Prints one JSON object.

    python tools/ref_scale.py [--pairs 1000000] [--genome-len 3100000000]

Runs on a GPU box only; everything lives in /dev/shm and is removed at the end."""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

EXE = os.path.join(ROOT, "urmap_b200", "bin", "urmap_b200")


def write_fasta(path, meta, seq):
    with open(path, "wb") as f:   # 60 columns, the layout index_build.fasta_bytes assumes
        for name, L, off in zip(meta["names"], meta["lens"], meta["offsets"]):
            f.write(b">" + name.encode() + b"\n")
            CH = 60 * (1 << 20)
            for o in range(0, L, CH):
                n = min(CH, L - o)
                s = seq[off + o:off + o + n].cpu().numpy()
                full = n // 60 * 60
                rows = np.empty((full // 60, 61), np.uint8)
                rows[:, :60] = s[:full].reshape(-1, 60)
                rows[:, 60] = 10
                f.write(rows.tobytes())
                if n > full:
                    f.write(s[full:].tobytes() + b"\n")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,memory.total", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return [l.strip() for l in q.stdout.splitlines() if l.strip()]


def run_map(args, gpus):
    """One `urmap_b200 -map2` run; returns its times and the peak device memory of the GPUs it used."""
    mon = subprocess.Popen(["nvidia-smi", "--query-gpu=index,memory.used", "--format=csv,noheader,nounits", "-lms", "50"],
                           stdout=subprocess.PIPE, text=True)
    try:
        t0 = time.time()
        p = subprocess.run([EXE] + args + ["-gpus", str(gpus), "-threads", str(os.cpu_count())], capture_output=True,
                           env=dict(os.environ, URMB_PROFILE="1"))
        wall = time.time() - t0
    finally:
        mon.terminate()
        samples = mon.communicate()[0]
    err = p.stderr.decode(errors="replace")
    if p.returncode != 0:
        raise RuntimeError(err[-800:])
    peak = {}
    for ln in samples.splitlines():
        f = [x.strip() for x in ln.split(",")]
        if len(f) == 2 and f[0].isdigit() and f[1].isdigit() and int(f[0]) < gpus:
            peak[int(f[0])] = max(peak.get(int(f[0]), 0), int(f[1]))
    m = re.search(r"load ([0-9.]+)s.*mapper total ([0-9.]+)s", err)
    out = {"wall_seconds": wall, "seconds_to_index_ready": float(m.group(1)), "seconds_in_mapper": float(m.group(2)),
           "peak_device_mib_per_gpu": [peak.get(g) for g in range(gpus)]}
    r = re.search(r"read ([0-9.]+) s, upload ([0-9.]+) s, parse ([0-9.]+) s \(kernels ([0-9.]+) s\), build ([0-9.]+) s", err)
    if r:
        out.update(read_seconds=float(r.group(1)), upload_seconds=float(r.group(2)), parse_seconds=float(r.group(3)),
                   parse_kernel_seconds=float(r.group(4)), build_seconds=float(r.group(5)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=1_000_000)
    ap.add_argument("--genome-len", type=int, default=3_100_000_000)
    ap.add_argument("--workdir", default="/dev/shm/urmb_ref_scale")
    a = ap.parse_args()
    import torch
    from urmap_b200 import build as BLD
    from urmap_b200 import gpu_synth
    BLD.build_engine()
    out = {"gpu": gpu_info(), "pairs": a.pairs, "genome_len": a.genome_len}
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    args = argparse.Namespace(genome_len=a.genome_len, pairs_per_step=1, read_len=150, sub=0.01, indel=0.001, single_end=False,
                              segdup_frac=0.03, tandem_frac=0.01)   # bench.py's genome
    meta, seq, blob = bench.build_workload(args, 0, 1, device)
    del blob
    os.makedirs(a.workdir, exist_ok=True)
    try:
        fa = os.path.join(a.workdir, "ref.fa")
        write_fasta(fa, meta, seq)
        out["fasta_bytes"] = os.path.getsize(fa)
        RL = 150
        r1, r2 = gpu_synth.sim_pe(seq, meta["lens"], meta["offsets"], a.pairs, device, RL, 0.01, 0.001, seed=7000)
        prefix = os.path.join(a.workdir, "reads")
        bench.write_fastq_pair(prefix, r1.cpu().numpy().reshape(-1), r2.cpu().numpy().reshape(-1), a.pairs, RL)
        del r1, r2, seq
        torch.cuda.empty_cache()
        ufi = os.path.join(a.workdir, "ref.ufi")
        t0 = time.time()
        subprocess.run([EXE, "-make_ufi", fa, "-output", ufi, "-gpu_build", "-quiet"], check=True)
        out["make_ufi_gpu_build_seconds"] = time.time() - t0
        out["ufi_bytes"] = os.path.getsize(ufi)
        reads = ["-map2", prefix + "_1.fq", "-reverse", prefix + "_2.fq"]
        sam_u, sam_r = os.path.join(a.workdir, "ufi.sam"), os.path.join(a.workdir, "ref.sam")
        ngpu = torch.cuda.device_count()
        for G in ([1, 8] if ngpu >= 8 else [1]):
            out[f"gpus_{G}"] = {
                "ufi": run_map(reads + ["-ufi", ufi, "-samout", sam_u], G),
                "ref": run_map(reads + ["-ref", fa, "-samout", sam_r], G),
            }
            out[f"gpus_{G}"]["sam_identity_ref_vs_ufi"] = bench.samdiff(sam_u, sam_r)
        r = out["gpus_1"]["ref"]
        peaks = bench.load_json("MEASURED_PEAKS.json")
        k = r.get("parse_kernel_seconds")
        if k:
            out["parse_kernel_input_gbs"] = out["fasta_bytes"] / k / 1e9
            # bytes the kernels move: the raw bytes read by four passes (header starts counted, then written; kept bytes
            # counted; scatter), SeqData written once
            moved = 4 * out["fasta_bytes"] + meta["seq_data_size"]
            out["parse_kernel_moved_gbs"] = moved / k / 1e9
            out["hbm_gbs_measured_peak"] = peaks.get("hbm_gbs")
            if peaks.get("hbm_gbs"):
                out["parse_kernel_share_of_hbm_peak"] = out["parse_kernel_moved_gbs"] / peaks["hbm_gbs"]
    finally:
        shutil.rmtree(a.workdir, ignore_errors=True)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
