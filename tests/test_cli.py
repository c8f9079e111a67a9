"""The drop-in command line (urmap_b200/bin/urmap_b200): URMAP's option spellings, UFI files and SAM output."""
import gzip
import os
import shutil
import subprocess

import pytest

from conftest import ROOT, expect, file_digest, have_gpu, make_ufi, sam_digest
from urmap_b200 import synth

BIN = os.path.join(ROOT, "urmap_b200", "bin", "urmap_b200")


@pytest.fixture(scope="module")
def cli(built_lib):
    assert os.path.exists(BIN)
    return BIN


def run(args, **kw):
    return subprocess.run(args, capture_output=True, text=True, **kw)


def test_make_ufi_is_byte_identical(cli, golden_dir, tmp_path):
    """-make_ufi (CPU builder) reproduces the reference's UFI file byte for byte (ufindex.cpp:83-408)."""
    make_ufi("golden", os.path.join(golden_dir, "ref.fa"), str(tmp_path / "ref.ufi"))


def test_make_ufi_options_match_reference(cli, golden_dir, tmp_path):
    fa = os.path.join(golden_dir, "ref.fa")
    for extra in (["-veryfast"], ["-maxix", "5", "-load_factor", "0.7"], ["-slots", "300007"], ["-wordlength", "20"]):
        make_ufi("golden" + "".join("_" + e.lstrip("-") for e in extra), fa, str(tmp_path / "a.ufi"), extra)


def test_invalid_command_lines(cli):
    r = run([cli, "-bogus", "1"])
    assert r.returncode == 1 and "Invalid command line" in r.stderr
    r = run([cli, "-ufi", "x.ufi"])
    assert r.returncode == 1 and "Invalid command line" in r.stderr
    r = run([cli, "-map2", "a.fq", "-ufi", "x.ufi"])
    assert r.returncode == 1 and "-reverse required" in r.stderr and "---Fatal error---" in r.stderr


@pytest.mark.skipif(have_gpu(), reason="checks the no-device failure mode")
def test_map_without_gpu_fails_loudly(cli, golden_dir, tmp_path):
    r = run([cli, "-map", os.path.join(golden_dir, "se.fq"), "-ufi", os.path.join(golden_dir, "ref.ufi"), "-samout",
             str(tmp_path / "o.sam")])
    assert r.returncode == 1 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("name,args", [
    ("se.sam", ["-map", "se.fq"]),
    ("se_veryfast.sam", ["-map", "se.fq", "-veryfast"]),
    ("pe.sam", ["-map2", "pe_1.fq", "-reverse", "pe_2.fq"]),
    ("pe_veryfast.sam", ["-map2", "pe_1.fq", "-reverse", "pe_2.fq", "-veryfast"]),
])
def test_cli_sam_matches_golden(cli, golden_dir, tmp_path, name, args):
    if not have_gpu():
        pytest.skip("no CUDA device")
    args = [os.path.join(golden_dir, a) if a.endswith(".fq") else a for a in args]
    out = tmp_path / name
    r = run([cli] + args + ["-ufi", os.path.join(golden_dir, "ref.ufi"), "-samout", str(out), "-threads", "4", "-batch", "97"])
    assert r.returncode == 0, r.stderr
    assert "Reads/sec" in r.stderr and "Mapped Q>=10" in r.stderr
    assert _unused(r.stderr) == []
    a = open(os.path.join(golden_dir, name), "rb").read().split(b"\n")
    b = open(out, "rb").read().split(b"\n")
    strip = lambda ls: [l for l in ls if not l.startswith(b"@PG")]
    assert strip(a) == strip(b)  # same records, same (input) order, same @SQ header


@pytest.mark.gpu
def test_cli_gz_input_and_gpu_built_index(cli, golden_dir, tmp_path):
    if not have_gpu():
        pytest.skip("no CUDA device")
    gz = tmp_path / "se.fq.gz"
    with open(os.path.join(golden_dir, "se.fq"), "rb") as f, gzip.open(gz, "wb") as g:
        shutil.copyfileobj(f, g)
    ufi = tmp_path / "gpu.ufi"
    r = run([cli, "-make_ufi", os.path.join(golden_dir, "ref.fa"), "-output", str(ufi), "-gpu_build", "-quiet"])
    assert r.returncode == 0, r.stderr
    assert open(ufi, "rb").read() == open(os.path.join(golden_dir, "ref.ufi"), "rb").read()   # the GPU builder is exact
    dense, dense_host = tmp_path / "dense.ufi", tmp_path / "dense_host.ufi"   # load factor 0.95: long links
    for out, extra in ((dense, ["-gpu_build"]), (dense_host, [])):
        r = run([cli, "-make_ufi", os.path.join(golden_dir, "ref.fa"), "-output", str(out), "-load_factor", "0.95", "-quiet"] + extra)
        assert r.returncode == 0, r.stderr
    assert open(dense, "rb").read() == open(dense_host, "rb").read()
    out = tmp_path / "o.sam"
    r = run([cli, "-map", str(gz), "-ufi", str(ufi), "-samout", str(out), "-quiet"])
    assert r.returncode == 0, r.stderr
    c = synth.compare_sam(os.path.join(golden_dir, "se.sam"), str(out))
    assert c["identical"] == c["total"] == 580 and c["header_equal"]


# ---- the block FASTQ reader (FASTQSeqSource::GetNextLo, fastqseqsource.cpp:9-116; linereader.cpp:54-99) on the CPU ----
def _fastq_records(path):
    """Plain restatement: CR bytes dropped everywhere, last line may lack LF, empty lines only at the end."""
    op = gzip.open if str(path).endswith(".gz") else open
    data = op(path, "rb").read().replace(b"\r", b"")
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    n_all = len(lines)
    while lines and lines[-1] == b"":
        lines.pop()
    if len(lines) % 4 and len(lines) + 4 - len(lines) % 4 <= n_all:   # empty sequence / quality lines of the last record
        lines += [b""] * (4 - len(lines) % 4)
    assert len(lines) % 4 == 0
    return [(lines[i][1:], lines[i + 1], lines[i + 3]) for i in range(0, len(lines), 4)]


def _dump(cli, fq, out, extra=()):
    r = run([cli, "-fastq_dump", str(fq), "-output", str(out)] + list(extra))
    assert r.returncode == 0, r.stderr
    return [tuple(l.split(b"\t")) for l in open(out, "rb").read().split(b"\n")[:-1]]


@pytest.mark.parametrize("variant", ["lf", "crlf", "no_final_lf", "trailing_blank", "gz", "ragged", "one", "empty_last",
                                     "empty_last_blank"])
def test_fastq_reader_matches_plain_parse(cli, golden_dir, tmp_path, variant):
    src = open(os.path.join(golden_dir, "se.fq"), "rb").read()
    fq = tmp_path / "in.fq"
    if variant == "crlf":
        src = src.replace(b"\n", b"\r\n")
    elif variant == "no_final_lf":
        src = src.rstrip(b"\n")
    elif variant == "trailing_blank":
        src = src + b"\n\n\n"
    elif variant == "ragged":   # reads of every length 0..150, labels with blanks
        recs = _fastq_records(os.path.join(golden_dir, "se.fq"))
        src = b"".join(b"@%s extra words\n%s\n+anything\n%s\n" % (l, s[:i % 151], q[:i % 151]) for i, (l, s, q) in enumerate(recs))
    elif variant == "one":
        src = b"@only\nACGT\n+\nIIII"
    elif variant == "empty_last":   # a last record with empty sequence and quality lines is a record (fastqseqsource.cpp:9-116)
        src = src + b"@r\n\n+\n\n"
    elif variant == "empty_last_blank":
        src = src + b"@r\n\n+\n\n\n\n"
    if variant == "gz":
        fq = tmp_path / "in.fq.gz"
        with gzip.open(fq, "wb") as g:
            g.write(src)
    else:
        fq.write_bytes(src)
    want = _fastq_records(fq)
    for extra in (["-batch", "1", "-threads", "1"], ["-batch", "7", "-threads", "3"], ["-batch", "97", "-threads", "8"],
                  ["-batch", "100000", "-threads", "5"]):
        if variant in ("ragged", "lf") or extra[1] != "1":
            assert _dump(cli, fq, tmp_path / "d.txt", extra) == want, (variant, extra)


def test_fastq_reader_pairs_and_errors(cli, golden_dir, tmp_path):
    g1, g2 = os.path.join(golden_dir, "pe_1.fq"), os.path.join(golden_dir, "pe_2.fq")
    got = _dump(cli, g1, tmp_path / "d.txt", ["-reverse", g2, "-batch", "33", "-threads", "4"])
    r1, r2 = _fastq_records(g1), _fastq_records(g2)
    assert got == [x for pair in zip(r1, r2) for x in pair]
    # mate files of different length (map2.cpp:31)
    short = tmp_path / "short.fq"
    short.write_bytes(b"".join(b"@%s\n%s\n+\n%s\n" % r for r in r2[:-3]))
    r = run([cli, "-fastq_dump", g1, "-reverse", str(short), "-output", str(tmp_path / "x"), "-batch", "50"])
    assert r.returncode == 1 and "Premature end of file in FASTQ2" in r.stderr
    good = b"@a\nACGT\n+\nIIII\n"
    for bad, msg in ((good + b"b\nACGT\n+\nIIII\n", "expected '@'"),
                     (good + b"@b\nACGT\n+\nIII\n", "4 bases, 3 quals"),
                     (good + b"@b x\nACGT\n+\nIII\n", "file %s label b x" % (tmp_path / "bad.fq")),
                     (good + b"@b\nAC-T\n+\nIIII\n", "Invalid sequence letter '-'"),
                     (good + b"@b\nAC\x01T\n+\nIIII\n", "Non-printing byte 0x01"),
                     (good + b"\n" + good, "Empty line nr 5"),
                     (good + b"@b\nACGT\n+\n", "Unexpected end-of-file")):
        f = tmp_path / "bad.fq"
        f.write_bytes(bad)
        for extra in (["-batch", "1"], ["-batch", "100", "-threads", "3"]):
            r = run([cli, "-fastq_dump", str(f), "-output", str(tmp_path / "x")] + extra)
            assert r.returncode == 1 and msg in r.stderr and "---Fatal error---" in r.stderr, (bad, extra, r.stderr)


def test_ufi_info_matches_reference(cli, oracle, golden_dir):
    """-ufi_info (ufistats.cpp:148-172): the same four lines (the reference prefixes its progress clock)."""
    ufi = os.path.join(golden_dir, "ref.ufi")
    r = run([cli, "-ufi_info", ufi])
    assert r.returncode == 0
    mine = [l.strip() for l in r.stderr.splitlines() if l.strip()]
    assert mine == ["Word length  24", "MaxIx  32", "SeqData  150064 (150.1kb)", "Slots  257171 (257.2kb)"]
    if os.path.exists(oracle.REF_BIN):
        ref = subprocess.run([oracle.REF_BIN, "-ufi_info", ufi], capture_output=True, text=True).stderr
        for l in mine:
            assert l in ref


# ---- -tabbedout (State2::OutputTab2, outputtab2.cpp:85-119): written by the formatter stage next to the SAM file ----
@pytest.mark.gpu
@pytest.mark.parametrize("name,extra", [("pe.tab", []), ("pe_veryfast.tab", ["-veryfast"])])
def test_cli_tabbedout_matches_golden(cli, golden_dir, tmp_path, name, extra):
    if not have_gpu():
        pytest.skip("no CUDA device")
    out, sam = tmp_path / name, tmp_path / "o.sam"
    r = run([cli, "-map2", os.path.join(golden_dir, "pe_1.fq"), "-reverse", os.path.join(golden_dir, "pe_2.fq"), "-ufi",
             os.path.join(golden_dir, "ref.ufi"), "-samout", str(sam), "-tabbedout", str(out), "-threads", "3", "-batch", "61"] + extra)
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == open(os.path.join(golden_dir, name), "rb").read()
    # the SAM file is the one written without -tabbedout
    c = synth.compare_sam(os.path.join(golden_dir, name.replace(".tab", ".sam")), str(sam))
    assert c["identical"] == c["total"] == 860


@pytest.mark.gpu
def test_cli_tabbedout_repeat_rich_vs_reference(cli, oracle, tmp_path):
    """Many second pairs: 2 Mb repeat-rich genome, 6 000 pairs (some mates damaged); the file equals the reference's
    (stored digest) and, where the reference binary has been built, the one it writes (-threads 1: input order)."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    g = synth.make_genome(2_000_000, n_contigs=4, seed=78, repeat_frac=0.15, n_runs=[(2, 0.3, 1500)], tandem=20, segdup=6)
    fa, ufi = str(tmp_path / "ref.fa"), str(tmp_path / "ref.ufi")
    g.write_fasta(fa)
    make_ufi("repeat_rich_2mb_seed78", fa, ufi)
    r1, r2, names = synth.sim_pe(g, 6000, 150, 0.02, 0.002, seed=5)
    r2 = r2.copy()
    r2[::40, :75] = r1[::40, :75]
    for path, arr, sfx in ((tmp_path / "r_1.fq", r1, b"/1"), (tmp_path / "r_2.fq", r2, b"/2")):
        with open(path, "wb") as f:
            for i in range(len(names)):
                s = arr[i].tobytes()
                f.write(b"@" + names[i] + b".%d" % i + sfx + b"\n" + s + b"\n+\n" + b"I" * len(s) + b"\n")
    args = ["-map2", str(tmp_path / "r_1.fq"), "-reverse", str(tmp_path / "r_2.fq"), "-ufi", ufi]
    r = run([cli] + args + ["-samout", str(tmp_path / "o.sam"), "-tabbedout", str(tmp_path / "o.tab"), "-batch", "1000"])
    assert r.returncode == 0, r.stderr
    got = open(tmp_path / "o.tab", "rb").read().split(b"\n")
    assert sum(1 for l in got if l and l.split(b"\t")[3] != b"*") > 100   # the case is exercised
    expect("tab/repeat_rich_2mb_seed78", file_digest(tmp_path / "o.tab"))
    if os.path.exists(oracle.REF_BIN):
        oracle.run_reference(args + ["-samout", str(tmp_path / "ref.sam"), "-tabbedout", str(tmp_path / "ref.tab"), "-threads", "1"])
        want = open(tmp_path / "ref.tab", "rb").read().split(b"\n")
        diff = [(a, b) for a, b in zip(want, got) if a != b]
        assert len(want) == len(got) and not diff, diff[:5]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pe", "se"])
def test_cli_two_gpus(cli, golden_dir, tmp_path, mode):
    """`-gpus 2` (SURVEY.md §8e through the drop-in itself): the index goes to GPU 0 over PCIe and on to GPU 1 over NVLink,
    batches alternate between the GPUs; the SAM file equals the golden one record for record, in input order."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    out = tmp_path / "o.sam"
    if mode == "pe":
        args = ["-map2", os.path.join(golden_dir, "pe_1.fq"), "-reverse", os.path.join(golden_dir, "pe_2.fq")]
        want, n = "pe.sam", 860
    else:
        args = ["-map", os.path.join(golden_dir, "se.fq")]
        want, n = "se.sam", 580
    r = run([cli] + args + ["-ufi", os.path.join(golden_dir, "ref.ufi"), "-samout", str(out), "-gpus", "2", "-batch", "37", "-threads", "4"])
    assert r.returncode == 0, r.stderr
    assert "2 GPU" in r.stderr
    c = synth.compare_sam(os.path.join(golden_dir, want), str(out))
    assert c["identical"] == c["total"] == n and c["header_equal"]
    one = tmp_path / "one.sam"
    r = run([cli] + args + ["-ufi", os.path.join(golden_dir, "ref.ufi"), "-samout", str(one), "-batch", "37", "-threads", "4"])
    assert r.returncode == 0, r.stderr
    strip = lambda p: [l for l in open(p, "rb").read().split(b"\n") if not l.startswith(b"@PG")]
    assert strip(out) == strip(one)   # same records in the same order


@pytest.mark.gpu
@pytest.mark.parametrize("contigs", [1, 3])
def test_cli_config1_gate(cli, oracle, tmp_path, contigs):
    """BASELINE.json configs[0] at its stated size: 5 000 000 bp of iid uniform ACGT (one contig, and the three-contig variant
    that exercises the contig padding and SetMappedPos), 100 000 x 150 bp single-end reads with 1 % substitutions and 0.1 %
    indels -- and the same number of read pairs.  The drop-in builds the index on the GPU (byte-identical to the reference's
    file) and maps from FASTQ files; its SAM files equal the reference's (stored digests), the oracle restatement's, and
    those of the reference binary (-threads 1: input order) where it has been built."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    g = synth.make_genome(5_000_000, n_contigs=contigs, seed=12345)
    fa, ufi, mine = str(tmp_path / "ref.fa"), str(tmp_path / "ref.ufi"), str(tmp_path / "mine.ufi")
    g.write_fasta(fa)
    make_ufi(f"config1_5mb_{contigs}_contigs", fa, ufi)
    r = run([cli, "-make_ufi", fa, "-output", mine, "-gpu_build", "-quiet"])
    assert r.returncode == 0, r.stderr
    assert open(mine, "rb").read() == open(ufi, "rb").read()
    ix = oracle.Index(ufi)
    reads, names = synth.sim_se(g, 100_000, 150, 0.01, 0.001, seed=777)
    fq = str(tmp_path / "se.fq")
    synth.write_fastq(fq, reads, names)
    b = oracle.ReadBatch.from_fastq(fq)
    res, runs = oracle.map_se(ix, b, threads=os.cpu_count())
    wants = [oracle.sam_header(ix) + oracle.sam_se(ix, b, res, runs)]
    got = str(tmp_path / "se.sam")
    if os.path.exists(oracle.REF_BIN):
        wants.append(str(tmp_path / "ref_se.sam"))
        oracle.run_reference(["-map", fq, "-ufi", ufi, "-samout", wants[-1], "-threads", "1"])
    r = run([cli, "-map", fq, "-ufi", mine, "-samout", got, "-quiet"])
    assert r.returncode == 0, r.stderr
    expect(f"sam/config1_5mb_{contigs}_contigs_se", sam_digest(got))
    for want in wants:
        c = synth.compare_sam(want, got)
        assert c["identical"] == c["total"] == 100_000 and c["header_equal"], c["diffs"][:5]
    r1, r2, names = synth.sim_pe(g, 100_000, 150, 0.01, 0.001, seed=778)
    f1, f2 = str(tmp_path / "p1.fq"), str(tmp_path / "p2.fq")
    synth.write_fastq(f1, r1, names, b"/1")
    synth.write_fastq(f2, r2, names, b"/2")
    b1, b2 = oracle.ReadBatch.from_fastq(f1), oracle.ReadBatch.from_fastq(f2)
    o1, o2, runs = oracle.map_pe(ix, b1, b2, threads=os.cpu_count())
    wants = [oracle.sam_header(ix) + oracle.sam_pe(ix, b1, b2, o1, o2, runs)]
    got = str(tmp_path / "pe.sam")
    if os.path.exists(oracle.REF_BIN):
        wants.append(str(tmp_path / "ref_pe.sam"))
        oracle.run_reference(["-map2", f1, "-reverse", f2, "-ufi", ufi, "-samout", wants[-1], "-threads", "1"])
    r = run([cli, "-map2", f1, "-reverse", f2, "-ufi", mine, "-samout", got, "-quiet"])
    assert r.returncode == 0, r.stderr
    expect(f"sam/config1_5mb_{contigs}_contigs_pe", sam_digest(got))
    for want in wants:
        c = synth.compare_sam(want, got)
        assert c["identical"] == c["total"] == 200_000 and c["header_equal"], c["diffs"][:5]
    ix.close()


@pytest.mark.gpu
def test_cli_contig_end_overhang(cli, oracle, tmp_path):
    """Pairs with a mate hanging 1 - 10 bases over either end of a contig: State1::SetMappedPos (state1.cpp:129-145) clears
    the top hit of such a mate, and OutputTab2 sees that cleared state only when a SAM file is written first
    (output2.cpp:10-16): the -tabbedout file differs with and without -samout.  Both forms, and the SAM file, equal the
    reference's (stored digests) and, where the reference binary has been built, the files it writes."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    import numpy as np
    g = synth.make_genome(600_000, n_contigs=3, seed=99)
    fa, ufi = str(tmp_path / "ref.fa"), str(tmp_path / "ref.ufi")
    g.write_fasta(fa)
    make_ufi("overhang_600kb_seed99", fa, ufi)
    rng = np.random.default_rng(5)
    comp = np.zeros(256, np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    rc = lambda x: comp[x[::-1]]
    r1, r2, names = [], [], []
    for c in range(3):
        off, L = int(g.offs[c]), int(g.lens[c])
        for hang in range(1, 11):
            for side in (0, 1):
                if c == 2 and side == 0:
                    continue   # past the end of the LAST contig the reference compares against bytes beyond its sequence buffer
                               # (extendpen.cpp:29-52 has no bound): undefined there, zero padding here
                tail = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=hang)
                if side == 0:   # right end of the contig: the reverse mate hangs over
                    a, b = g.asc[off + L - 450: off + L - 300].copy(), rc(np.concatenate([g.asc[off + L - (150 - hang): off + L], tail]))
                else:           # left end: the forward mate starts before the contig
                    a, b = np.concatenate([tail, g.asc[off: off + 150 - hang]]), rc(g.asc[off + 300: off + 450].copy())
                if len(names) % 2:
                    a, b = b, a
                r1.append(a)
                r2.append(b)
                names.append(b"ov%d_c%d_h%d_s%d" % (len(names), c, hang, side))
    f1, f2 = str(tmp_path / "p1.fq"), str(tmp_path / "p2.fq")
    synth.write_fastq(f1, np.array(r1), names, b"/1")
    synth.write_fastq(f2, np.array(r2), names, b"/2")
    args = ["-map2", f1, "-reverse", f2, "-ufi", ufi]
    p = lambda n: str(tmp_path / n)
    r = run([cli] + args + ["-samout", p("o.sam"), "-tabbedout", p("o_a.tab"), "-batch", "16", "-quiet"])
    assert r.returncode == 0, r.stderr
    r = run([cli] + args + ["-tabbedout", p("o_b.tab"), "-batch", "16", "-quiet"])
    assert r.returncode == 0, r.stderr
    assert open(p("o_a.tab"), "rb").read() != open(p("o_b.tab"), "rb").read()   # the case is what it claims to be
    expect("tab/overhang_600kb_seed99_with_samout", file_digest(p("o_a.tab")))
    expect("tab/overhang_600kb_seed99_without_samout", file_digest(p("o_b.tab")))
    expect("sam/overhang_600kb_seed99", sam_digest(p("o.sam")))
    assert sam_digest(p("o.sam"))["records"] == 2 * len(names)
    if os.path.exists(oracle.REF_BIN):
        oracle.run_reference(args + ["-threads", "1", "-samout", p("ref.sam"), "-tabbedout", p("ref_a.tab")])
        oracle.run_reference(args + ["-threads", "1", "-tabbedout", p("ref_b.tab")])
        assert open(p("o_a.tab"), "rb").read() == open(p("ref_a.tab"), "rb").read()
        assert open(p("o_b.tab"), "rb").read() == open(p("ref_b.tab"), "rb").read()
        c = synth.compare_sam(p("ref.sam"), p("o.sam"))
        assert c["identical"] == c["total"] == 2 * len(names) and c["header_equal"], c["diffs"][:5]


def test_ufi_validate(cli, oracle, golden_dir, tmp_path):
    """-ufi_validate and -make_ufi ... -validate (cmd_ufi_validate ufistats.cpp:141-146, UFIndex::Validate ufindex.cpp:611-658):
    silent success on consistent tables -- the golden one and a dense one full of long links -- and the reference's fatal
    "WordToSlot != Slot" on a table with one stored position moved (the reference binary judges the same file the same way)."""
    import struct
    golden = os.path.join(golden_dir, "ref.ufi")
    r = run([cli, "-ufi_validate", golden, "-quiet"])
    assert r.returncode == 0, r.stderr
    dense = str(tmp_path / "dense.ufi")
    r = run([cli, "-make_ufi", os.path.join(golden_dir, "ref.fa"), "-output", dense, "-load_factor", "0.95", "-validate", "-quiet"])
    assert r.returncode == 0, r.stderr
    raw = open(dense, "rb").read()
    hdr = raw.index(struct.pack("<I", 0x55464932)) + 4
    slots = struct.unpack_from("<Q", raw, 16)[0]
    tallies = raw[hdr:hdr + 5 * slots:5]
    assert tallies.count(bytes([125])) > 100   # long links are there
    r = run([cli, "-ufi_validate", dense, "-quiet", "-threads", "3"])
    assert r.returncode == 0, r.stderr
    # move the position stored in the first BOTH1 slot by one base: its 24-mer no longer hashes to the slot
    raw = bytearray(open(golden, "rb").read())
    hdr = raw.index(struct.pack("<I", 0x55464932)) + 4
    slots = struct.unpack_from("<Q", raw, 16)[0]
    s = next(i for i in range(slots) if raw[hdr + 5 * i] == 255)
    pos = struct.unpack_from("<I", raw, hdr + 5 * s + 1)[0]
    struct.pack_into("<I", raw, hdr + 5 * s + 1, pos + 1)
    bad = str(tmp_path / "bad.ufi")
    open(bad, "wb").write(raw)
    r = run([cli, "-ufi_validate", bad])
    assert r.returncode == 1 and "---Fatal error---" in r.stderr and "WordToSlot != Slot" in r.stderr
    if os.path.exists(oracle.REF_BIN):
        import subprocess
        for path, ok in ((golden, True), (dense, True), (bad, False)):
            p = subprocess.run([oracle.REF_BIN, "-ufi_validate", path, "-quiet"], capture_output=True, text=True)
            assert (p.returncode == 0) == ok
            if not ok:
                assert "WordToSlot != Slot" in p.stderr


def test_args_file(cli, golden_dir, tmp_path):
    """`file: args.txt` on the command line stands for the fields of that file, '#' starts a comment (cmdline.cpp:40-56,162-179)."""
    args = tmp_path / "args.txt"
    out = tmp_path / "o.ufi"
    args.write_text("-make_ufi %s   # the reference\n\n  -output %s\n-quiet\n" % (os.path.join(golden_dir, "ref.fa"), out))
    r = run([cli, "file:", str(args)])
    assert r.returncode == 0, r.stderr
    assert open(out, "rb").read() == open(os.path.join(golden_dir, "ref.ufi"), "rb").read()
    r = run([cli, "-ufi_info", "file:", str(args)])   # "-ufi_info -make_ufi ...": two commands
    assert r.returncode == 1 and "Invalid command line" in r.stderr


def _unused(stderr):
    return [l.split("Option -")[1].split()[0] for l in stderr.splitlines() if "WARNING: Option -" in l and "not used" in l]


@pytest.mark.parametrize("cmd", ["make_ufi", "ufi_info", "ufi_validate"])
def test_unused_option_warnings(cli, oracle, golden_dir, tmp_path, cmd):
    """CheckUsedOpts (cmdline.cpp:13-26): an option that was given but that the command never looks at is named in a warning
    after the command has run, in the order of myopts.h -- the same names in the same order as the reference binary prints
    (this program uses -threads for -ufi_validate, the one deliberate difference).  The reference's names are stored."""
    import subprocess
    g = golden_dir
    base = {"make_ufi": ["-make_ufi", os.path.join(g, "ref.fa"), "-output", str(tmp_path / "o.ufi")],
            "ufi_info": ["-ufi_info", os.path.join(g, "ref.ufi")],
            "ufi_validate": ["-ufi_validate", os.path.join(g, "ref.ufi")]}[cmd]
    extras = ["-veryfast", "-minq", "7", "-reverse", os.path.join(g, "pe_2.fq"), "-threads", "2", "-maxix", "32", "-validate",
              "-load_factor", "0.6", "-wordlength", "24", "-ufi", os.path.join(g, "ref.ufi"), "-samout", str(tmp_path / "x.sam")]
    if cmd == "make_ufi":
        extras = [e for e in extras if e not in ("-maxix", "32", "-wordlength", "24", "-load_factor", "0.6", "-validate")] + ["-validate"]
    mine = run([cli] + base + extras)
    assert mine.returncode == 0, mine.stderr[-300:]
    got = _unused(mine.stderr)
    expect("unused_options/" + cmd, got)   # for -ufi_validate: the reference's names but -threads
    if os.path.exists(oracle.REF_BIN):
        ref = subprocess.run([oracle.REF_BIN] + base + extras, capture_output=True, text=True)
        assert ref.returncode == 0, ref.stderr[-300:]
        want = _unused(ref.stderr)
        if cmd == "ufi_validate":
            want = [w for w in want if w != "threads"]
        assert got == want
    assert len(got) >= 3


@pytest.mark.gpu
def test_cli_unused_options_map(cli, golden_dir, tmp_path):
    """-map looks at neither -minq nor -load_factor, -map2 looks at -minq (probed on the reference binary): the warnings come
    after the run, in the order of myopts.h; the log file ends with the reference's Finished / Elapsed time / Max memory lines."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    ufi = os.path.join(golden_dir, "ref.ufi")
    log = tmp_path / "run.log"
    r = run([cli, "-map", os.path.join(golden_dir, "se.fq"), "-ufi", ufi, "-samout", str(tmp_path / "a.sam"), "-load_factor", "0.6",
             "-minq", "7", "-log", str(log)])
    assert r.returncode == 0, r.stderr
    assert _unused(r.stderr) == ["minq", "load_factor"]
    text = log.read_text()
    assert "Started " in text and "Finished " in text and "Elapsed time " in text and "Option -minq not used" in text
    r = run([cli, "-map2", os.path.join(golden_dir, "pe_1.fq"), "-reverse", os.path.join(golden_dir, "pe_2.fq"), "-ufi", ufi,
             "-samout", str(tmp_path / "b.sam"), "-minq", "7", "-maxix", "32"])
    assert r.returncode == 0, r.stderr
    assert _unused(r.stderr) == ["maxix"]
