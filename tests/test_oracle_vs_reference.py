"""Pins the oracle restatement against the UNMODIFIED reference binary on fresh seeded data: its SAM files equal the
reference's (stored digests, tests/golden/reference_outputs.json) and, where the binary has been built (oracle/_ref/urmap,
from the reference's sources by oracle/Makefile), the files it writes at test time."""
import os

import pytest

from conftest import expect, make_ufi, sam_digest
from urmap_b200 import synth


@pytest.fixture(scope="module")
def ref_env(oracle, built_lib, tmp_path_factory):
    d = tmp_path_factory.mktemp("refenv")
    g = synth.make_genome(1_000_000, n_contigs=2, seed=31, repeat_frac=0.05, n_runs=[(0, 0.3, 500)], tandem=4)
    fa, ufi = str(d / "ref.fa"), str(d / "ref.ufi")
    g.write_fasta(fa)
    make_ufi("ovr_1mb_seed31", fa, ufi)
    return d, g, ufi


def _check(oracle, key, mine, ref_args, sam, n):
    assert sam_digest(mine)["records"] == n
    expect("sam/" + key, sam_digest(mine))
    if os.path.exists(oracle.REF_BIN):
        oracle.run_reference(ref_args + ["-samout", sam, "-threads", "1"])
        c = synth.compare_sam(sam, mine)
        assert c["identical"] == c["total"] == n and c["header_equal"], c["diffs"][:5]


@pytest.mark.parametrize("sub,indel,veryfast", [(0.01, 0.001, False), (0.05, 0.01, False), (0.02, 0.002, True)])
def test_se_matches_reference(oracle, ref_env, sub, indel, veryfast):
    d, g, ufi = ref_env
    reads, names = synth.sim_se(g, 4000, 150, sub, indel, seed=int(sub * 1000) + 5)
    fq, sam = str(d / "se.fq"), str(d / "se.sam")
    synth.write_fastq(fq, reads, names)
    ix = oracle.Index(ufi)
    b = oracle.ReadBatch.from_fastq(fq)
    res, runs = oracle.map_se(ix, b, method=7 if veryfast else 6, threads=4)
    mine = oracle.sam_header(ix) + oracle.sam_se(ix, b, res, runs)
    _check(oracle, f"ovr_se_{sub}_{indel}{'_veryfast' if veryfast else ''}", mine,
           ["-map", fq, "-ufi", ufi] + (["-veryfast"] if veryfast else []), sam, 4000)


@pytest.mark.parametrize("sub,indel,veryfast,rl", [(0.01, 0.001, False, 150), (0.05, 0.01, False, 150), (0.02, 0.002, True, 150),
                                                   (0.02, 0.002, False, 250)])
def test_pe_matches_reference(oracle, ref_env, sub, indel, veryfast, rl):
    d, g, ufi = ref_env
    r1, r2, names = synth.sim_pe(g, 3000, rl, sub, indel, seed=int(sub * 1000) + 7)
    f1, f2, sam = str(d / "p1.fq"), str(d / "p2.fq"), str(d / "pe.sam")
    synth.write_fastq(f1, r1, names, b"/1")
    synth.write_fastq(f2, r2, names, b"/2")
    ix = oracle.Index(ufi)
    b1, b2 = oracle.ReadBatch.from_fastq(f1), oracle.ReadBatch.from_fastq(f2)
    o1, o2, runs = oracle.map_pe(ix, b1, b2, pe_method=5 if veryfast else 4, threads=4)
    mine = oracle.sam_header(ix) + oracle.sam_pe(ix, b1, b2, o1, o2, runs)
    _check(oracle, f"ovr_pe_{rl}_{sub}_{indel}{'_veryfast' if veryfast else ''}", mine,
           ["-map2", f1, "-reverse", f2, "-ufi", ufi] + (["-veryfast"] if veryfast else []), sam, 6000)


def test_maxix_above_32_matches_reference(oracle, built_lib, tmp_path):
    """-maxix 100 (ufindexio.cpp:135-136): the reference indexes and walks lists of up to 100 positions; the restatement's
    rows follow (repeat-rich genome with tandem arrays, single-end and paired)."""
    g = synth.make_genome(300_000, n_contigs=2, seed=78, repeat_frac=0.35, n_runs=[(0, 0.3, 300)], tandem=12)
    fa, ufi = str(tmp_path / "m.fa"), str(tmp_path / "m.ufi")
    g.write_fasta(fa)
    make_ufi("ovr_300kb_seed78_maxix_100", fa, ufi, ["-maxix", "100"])
    ix = oracle.Index(ufi)
    assert ix.max_ix == 100
    reads, names = synth.sim_se(g, 1500, 150, 0.02, 0.002, seed=5)
    fq, sam = str(tmp_path / "se.fq"), str(tmp_path / "se.sam")
    synth.write_fastq(fq, reads, names)
    b = oracle.ReadBatch.from_fastq(fq)
    res, runs = oracle.map_se(ix, b, threads=4)
    _check(oracle, "ovr_maxix_100_se", oracle.sam_header(ix) + oracle.sam_se(ix, b, res, runs), ["-map", fq, "-ufi", ufi],
           sam, 1500)
    r1, r2, names = synth.sim_pe(g, 1000, 150, 0.02, 0.002, seed=15)
    f1, f2, sam2 = str(tmp_path / "p1.fq"), str(tmp_path / "p2.fq"), str(tmp_path / "pe.sam")
    synth.write_fastq(f1, r1, names, b"/1")
    synth.write_fastq(f2, r2, names, b"/2")
    b1, b2 = oracle.ReadBatch.from_fastq(f1), oracle.ReadBatch.from_fastq(f2)
    o1, o2, runs = oracle.map_pe(ix, b1, b2, threads=4)
    _check(oracle, "ovr_maxix_100_pe", oracle.sam_header(ix) + oracle.sam_pe(ix, b1, b2, o1, o2, runs),
           ["-map2", f1, "-reverse", f2, "-ufi", ufi], sam2, 2000)
    ix.close()
