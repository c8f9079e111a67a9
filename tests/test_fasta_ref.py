"""Mapping straight from a FASTA reference (-ref): the parse kernels (urmap_b200/csrc/urmb_fasta.cu) must give exactly the
SeqData, labels, lengths and offsets of the UFI file the host -make_ufi writes (UfiBuilder::ReadFasta), and -ref must map
exactly as -ufi with the table -make_ufi builds for the same options."""
import gzip
import os
import re
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

from conftest import CLI, ROOT, have_gpu

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))

GOLDEN = os.path.join(ROOT, "tests", "golden")
TILE = 16384   # bytes one warp of the parse kernels reads


def _ufi_sections(path):
    """(records [(label bytes, length, offset)], SeqData) of a UFI file (ufindexio.cpp:15-49)."""
    raw = open(path, "rb").read()
    _, _, _, seq_size, slots, n = struct.unpack_from("<IIIIQI", raw, 0)
    o, recs = 28, []
    for _ in range(n):
        ln, off, nl = struct.unpack_from("<III", raw, o)
        recs.append((raw[o + 12:o + 12 + nl], ln, off))
        o += 12 + nl
    o += 4 + 5 * slots + 4
    return recs, raw[o:o + seq_size], raw


def _blob(raw, slots):
    o = raw.index(struct.pack("<I", 0x55464932)) + 4
    return raw[o:o + 5 * slots]


def _edge_cases():
    rng = np.random.default_rng(5)
    acgt = lambda n: bytes(rng.choice(np.frombuffer(b"ACGTacgtN", np.uint8), n))
    lines = lambda s, w=60: b"".join(s[i:i + w] + b"\n" for i in range(0, len(s), w))
    c = {
        "lf": b">chr1 first contig\nACGTacgt\nNNNN\n>chr2\nGGG\n",
        "crlf": b">chr1 first contig\r\nACGTacgt\r\nNNNN\r\n>chr2\r\nGGG\r\n",
        "cr_inside": b">ch\rr1\r desc\r\nAC\rGT\r\r\n>c2\rx\nG\rG\n\r\r>c3\nTT\n",
        "junk_in_sequence": b">s\nacgtRYKMswbdhvn 0123*-.\tAC\x80\xff\xe9gt\x00\x7fz{@[`\n",
        "blank_lines_first": b"\n\r\n\r\r\n\n>a\nAC\n",
        "empty_label_and_tab": b">\nACGT\n>x\ty z\nGG\n>\t\nTT\n",
        "empty_records": b">e1\n>a\nAC\n>e2\n\n>e3\n--..**\n>b\nGT\n>e4\n>e5\n\r\n",
        "empty_only": b">e1\n\n>e2\n",
        "no_final_lf": b">a\nACGT\n>b\nGG",
        "no_final_lf_cr": b">a\nACGT\n>b\nGG\r",
        "gt_in_sequence": b">a\nAC>GT\n \t>x\nGG\n\r>y\nTT\n>z>w\nA>\n",
        "one_long_line": b">big\n" + acgt(3_000_000) + b"\n>tail\nAC\n",
        "tiny_records": b"".join(b">r%d\n%s\n" % (i, b"ACGT"[: i % 5]) for i in range(3000)),
        "spanning_records": b"".join(b">c%d\n" % i + lines(acgt(n)) for i, n in enumerate((70_000, 5, 40_000, 33_000))),
        "header_at_tile": b">a\n" + b"A" * (TILE - 4) + b"\n>b\nGG\n",
        "cr_across_tile": b">a\n" + b"C" * (TILE - 6) + b"\n\r\r>b\nGG\n",
        "header_line_across_tile": b">a\nAC\n>b " + b"d" * (3 * TILE) + b"\nTT\n",
        "empty": b"",
        "err_line1": b"ACGT\n>a\nAC\n",
        "err_line3": b"\n\r\n  \n>a\nAC\n",
        "err_cr_line": b"\r\n\rx\n>a\nA",
        "err_no_header": b"acgt",
        "err_late": b"\n" * 70_000 + b"x\n>a\nA\n",
    }
    return c


def _fuzz_cases(n=300, seed=2024):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b">>\n\n\n\r\r  \tACGTacgtNnRy-.*0\x00\xff", np.uint8)
    out = []
    for i in range(n):
        size = int(rng.integers(0, 400)) if i % 25 else int(rng.integers(TILE - 200, 2 * TILE + 200))
        data = bytes(rng.choice(alpha, size))
        if i % 3 == 0:
            data = b">" + data
        out.append(data)
    return out


def _host_parse(tmp_path, data):
    """-make_ufi on the CPU: (returncode, stderr bytes, records, SeqData)."""
    fa = str(tmp_path / "x.fa")
    with open(fa, "wb") as f:
        f.write(data)
    out = str(tmp_path / "x.ufi")
    r = subprocess.run([CLI, "-make_ufi", fa, "-output", out, "-quiet"], capture_output=True)
    if r.returncode != 0:
        return r.returncode, r.stderr, fa, None, None
    recs, seq, _ = _ufi_sections(out)
    return 0, r.stderr, fa, recs, seq


def _check_against_host(tmp_path, data):
    import emu_fasta_py
    rc, seq, recs, dropped, err = emu_fasta_py.emu_parse_fasta(data)
    hrc, stderr, fa, hrecs, hseq = _host_parse(tmp_path, data)
    if hrc != 0:
        assert rc == -2, (rc, stderr)   # URMB_E_IO
        assert ("Bad FASTA file %s, %s" % (fa, err)).encode() in stderr, (err, stderr[-300:])
        return "error"
    assert rc == 0, err
    assert seq == hseq
    assert recs == hrecs
    warned = re.findall(rb"WARNING: Empty sequence in FASTA file [^\n]*?, label >([^\n]*)\n", stderr)
    assert [d.split(b"\0")[0] for d in dropped] == warned   # printed with %s
    return "ok"


@pytest.fixture(scope="module")
def cli(built_lib):
    assert os.path.exists(CLI)
    return CLI


@pytest.mark.parametrize("name", sorted(_edge_cases()))
def test_emulated_parse_edge_cases(cli, tmp_path, name):
    kind = _check_against_host(tmp_path, _edge_cases()[name])
    assert kind == ("error" if name.startswith("err_") else "ok")


def test_emulated_parse_fuzz(cli, tmp_path):
    kinds = [_check_against_host(tmp_path, d) for d in _fuzz_cases()]
    assert kinds.count("ok") > 50 and kinds.count("error") > 50


def test_emulated_parse_golden_reference(cli, golden_dir, tmp_path):
    import emu_fasta_py
    data = open(os.path.join(golden_dir, "ref.fa"), "rb").read()
    rc, seq, recs, dropped, _ = emu_fasta_py.emu_parse_fasta(data)
    want_recs, want_seq, _ = _ufi_sections(os.path.join(golden_dir, "ref.ufi"))
    assert rc == 0 and seq == want_seq and recs == want_recs and dropped == []


def test_ref_and_ufi_are_exclusive(cli, tmp_path):
    fa = os.path.join(GOLDEN, "ref.fa")
    r = subprocess.run([cli, "-map", os.path.join(GOLDEN, "se.fq"), "-ref", fa, "-ufi", "x.ufi", "-samout", str(tmp_path / "a.sam")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "-ufi and -ref are mutually exclusive" in r.stderr
    r = subprocess.run([cli, "-map", os.path.join(GOLDEN, "se.fq"), "-samout", str(tmp_path / "a.sam")], capture_output=True, text=True)
    assert r.returncode == 1 and "-ufi required" in r.stderr


# ---------------------------------------------------------------- GPU ----------------------------------------------------

def _run(args):
    return subprocess.run(args, capture_output=True, text=True)


def _strip_pg(path):
    return [l for l in open(path, "rb").read().split(b"\n") if not l.startswith(b"@PG")]


def _unused(stderr):
    return [l.split("Option -")[1].split()[0] for l in stderr.splitlines() if "WARNING: Option -" in l and "not used" in l]


@pytest.mark.gpu
@pytest.mark.parametrize("name,args", [
    ("se.sam", ["-map", "se.fq"]),
    ("se_veryfast.sam", ["-map", "se.fq", "-veryfast", "-maxix", "32"]),
    ("pe.sam", ["-map2", "pe_1.fq", "-reverse", "pe_2.fq"]),
    ("pe_veryfast.sam", ["-map2", "pe_1.fq", "-reverse", "pe_2.fq", "-veryfast", "-maxix", "32"]),
    ("pe.tab", ["-map2", "pe_1.fq", "-reverse", "pe_2.fq"]),
    ("pe_veryfast.tab", ["-map2", "pe_1.fq", "-reverse", "pe_2.fq", "-veryfast", "-maxix", "32"]),
])
@pytest.mark.parametrize("gz", [False, True])
def test_ref_matches_golden(cli, golden_dir, tmp_path, name, args, gz):
    """-ref tests/golden/ref.fa (plain or gzip) reproduces the reference's golden SAM and -tabbedout files."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    fa = os.path.join(golden_dir, "ref.fa")
    if gz:   # the slot count follows the size of the file on disk, as for -make_ufi: give the plain file's table
        fa = str(tmp_path / "ref.fa.gz")
        with open(os.path.join(golden_dir, "ref.fa"), "rb") as f, gzip.open(fa, "wb") as g:
            shutil.copyfileobj(f, g)
        slots = struct.unpack_from("<Q", open(os.path.join(golden_dir, "ref.ufi"), "rb").read(24), 16)[0]
        args = args + ["-slots", str(slots)]
    args = [os.path.join(golden_dir, a) if a.endswith(".fq") else a for a in args]
    sam, tab = tmp_path / "o.sam", tmp_path / "o.tab"
    extra = ["-tabbedout", str(tab)] if name.endswith(".tab") else []
    r = _run([cli] + args + ["-ref", fa, "-samout", str(sam), "-threads", "4", "-batch", "97"] + extra)
    assert r.returncode == 0, r.stderr
    assert "parse" in r.stderr and "build" in r.stderr and _unused(r.stderr) == []
    if name.endswith(".tab"):
        assert open(tab, "rb").read() == open(os.path.join(golden_dir, name), "rb").read()
        name = name.replace(".tab", ".sam")
    assert _strip_pg(sam) == _strip_pg(os.path.join(golden_dir, name))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pe", "se"])
def test_ref_two_gpus(cli, golden_dir, tmp_path, mode):
    """-ref with -gpus 2: the FASTA bytes go to both GPUs, each parses and builds; the SAM file equals the golden one."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    g = golden_dir
    args = (["-map2", os.path.join(g, "pe_1.fq"), "-reverse", os.path.join(g, "pe_2.fq")] if mode == "pe"
            else ["-map", os.path.join(g, "se.fq")])
    out = tmp_path / "o.sam"
    r = _run([cli] + args + ["-ref", os.path.join(g, "ref.fa"), "-samout", str(out), "-gpus", "2", "-batch", "37", "-threads", "4"])
    assert r.returncode == 0, r.stderr
    assert "2 GPU" in r.stderr
    assert _strip_pg(out) == _strip_pg(os.path.join(g, "pe.sam" if mode == "pe" else "se.sam"))


def _device_bytes(ptr, n):
    import torch

    class _Dev:   # a device buffer owned by the engine, seen through the CUDA array interface
        __cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (ptr, False), "version": 3}

    return torch.as_tensor(_Dev(), device="cuda").cpu().numpy().tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [["-veryfast"], ["-wordlength", "20", "-maxix", "5"], ["-load_factor", "0.8"]])
def test_ref_repeat_rich_matches_make_ufi(cli, tmp_path, extra):
    """On the repeat-rich 400 kb genome of test_index_build.py the device table and SeqData equal the -make_ufi file's
    sections byte for byte, and -ref maps exactly as -ufi."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    from urmap_b200 import engine, synth
    g = synth.make_genome(400_000, n_contigs=3, seed=31, repeat_frac=0.15, n_runs=[(1, 0.3, 900)], tandem=15, segdup=4)
    fa, ufi = str(tmp_path / "r.fa"), str(tmp_path / "r.ufi")
    g.write_fasta(fa)
    r = _run([cli, "-make_ufi", fa, "-output", ufi, "-quiet"] + extra)
    assert r.returncode == 0, r.stderr
    recs, seq, raw = _ufi_sections(ufi)
    wl = int(extra[extra.index("-wordlength") + 1]) if "-wordlength" in extra else 24
    mx = int(extra[extra.index("-maxix") + 1]) if "-maxix" in extra else (3 if "-veryfast" in extra else 32)
    lf = float(extra[extra.index("-load_factor") + 1]) if "-load_factor" in extra else 0.6
    ctx = engine.Context(0)
    contigs = ctx.index_from_fasta(fa, word_length=wl, max_ix=mx, load_factor=lf)
    assert contigs == [(l.decode(), n, o) for l, n, o in recs]
    d = ctx.device_index()
    slots = struct.unpack_from("<Q", raw, 16)[0]
    assert (d.word_length, d.max_ix, d.seq_data_size, d.slot_count) == (wl, mx, len(seq), slots)
    assert _device_bytes(d.d_seq, len(seq) + 4096) == seq + bytes(4096)
    assert _device_bytes(d.d_blob, 5 * slots) == _blob(raw, slots)
    ctx.close()
    reads, names = synth.sim_se(g, 3000, 150, 0.02, 0.002, seed=8)
    fq = str(tmp_path / "r.fq")
    synth.write_fastq(fq, reads, names)
    sams = []
    for src in (["-ufi", ufi], ["-ref", fa]):
        out = str(tmp_path / ("a%d.sam" % len(sams)))
        r = _run([cli, "-map", fq, "-samout", out, "-threads", "4"] + src + (extra if src[0] == "-ref" else
                                                                              [e for e in extra if e == "-veryfast"]))
        assert r.returncode == 0, r.stderr
        sams.append(_strip_pg(out))
    assert sams[0] == sams[1]


@pytest.mark.gpu
def test_parse_on_gpu_matches_emulator(built_lib, tmp_path):
    """The edge-case FASTA files parsed on the GPU give the SeqData the emulated kernels give."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    import emu_fasta_py
    from urmap_b200 import engine
    ctx = engine.Context(0)
    n = 0
    for name, data in sorted(_edge_cases().items()):
        rc, seq, recs, dropped, err = emu_fasta_py.emu_parse_fasta(data)
        fa = str(tmp_path / "e.fa")
        with open(fa, "wb") as f:
            f.write(data)
        if rc != 0 or not seq:
            with pytest.raises(engine.UrmbError) as e:
                ctx.index_from_fasta(fa)
            assert e.value.code == -2 and (err in str(e.value) if err else "no sequence" in str(e.value)), (name, str(e.value))
            continue
        contigs = ctx.index_from_fasta(fa)
        d = ctx.device_index()
        assert _device_bytes(d.d_seq, len(seq) + 4096) == seq + bytes(4096), name
        assert [(c[1], c[2]) for c in contigs] == [(r[1], r[2]) for r in recs], name
        assert ctx.dropped == [x.split(b"\0")[0].decode() for x in dropped], name
        n += 1
    assert n >= 15
    ctx.close()


@pytest.mark.gpu
def test_ref_builder_refusal(cli, golden_dir, tmp_path):
    """-maxix above 254 is refused by the GPU builder: -ref exits 1 with its message and points to -make_ufi."""
    if not have_gpu():
        pytest.skip("no CUDA device")
    r = _run([cli, "-map", os.path.join(golden_dir, "se.fq"), "-ref", os.path.join(golden_dir, "ref.fa"), "-samout",
              str(tmp_path / "a.sam"), "-maxix", "300"])
    assert r.returncode == 1 and "-maxix above 254" in r.stderr and "-make_ufi" in r.stderr, r.stderr
