"""GPU parity tests proper: every call goes through the C-ABI (liburmb.so) and is compared, bit for bit, with
the oracle restatement and with the golden SAMs of the unmodified reference.  Integer / index work only:
the bar is exact equality (positions, strand, scores, MAPQ, path runs => CIGAR)."""
import os

import numpy as np
import pytest

from conftest import CLI, have_gpu, make_ufi
from urmap_b200 import synth

pytestmark = pytest.mark.gpu

FIELDS = ("db_pos", "score", "best", "second", "mapq", "flags", "hit_count", "hsp_count")


def _paths(res, runs):
    return [tuple(runs[r["path_off"]:r["path_off"] + r["path_runs"]].tolist()) for r in res]


def assert_same(ro, uo, rg, ug):
    assert len(ro) == len(rg)
    for f in FIELDS:
        bad = np.nonzero(ro[f] != rg[f])[0]
        assert len(bad) == 0, (f, bad[:5], ro[bad[:3]], rg[bad[:3]])
    assert _paths(ro, uo) == _paths(rg, ug)


def canon(res, runs):
    """Results with path offsets replaced by the path itself (pool layout is not deterministic)."""
    return [tuple(int(r[f]) for f in FIELDS) + (p,) for r, p in zip(res, _paths(res, runs))]


@pytest.fixture(scope="module")
def eng(built_lib):
    if not have_gpu():
        pytest.skip("no CUDA device")
    return built_lib


@pytest.fixture(scope="module")
def golden_ctxs(eng, golden_dir):
    hix = eng.HostIndex(os.path.join(golden_dir, "ref.ufi"))
    ctxs = {}
    for key, kw in (("se", {}), ("se_veryfast", {"method": 7}), ("pe", {}), ("pe_veryfast", {"pe_method": 5})):
        c = eng.Context(0, **kw)
        c.set_index(hix)
        ctxs[key] = c
    yield ctxs
    for c in ctxs.values():
        c.close()


@pytest.mark.parametrize("key", ["se", "se_veryfast"])
def test_golden_se(eng, oracle, golden_oix, golden_dir, golden_ctxs, key):
    b = oracle.ReadBatch.from_fastq(os.path.join(golden_dir, "se.fq"))
    res, runs = golden_ctxs[key].map_se(b.seqs, b.offs)
    ro, uo = oracle.map_se(golden_oix, b, method=7 if key.endswith("veryfast") else 6)
    assert_same(ro, uo, res, runs)
    sam = oracle.sam_header(golden_oix) + oracle.sam_se(golden_oix, b, res, runs)
    c = synth.compare_sam(os.path.join(golden_dir, key + ".sam"), sam)
    assert c["identical"] == c["total"] == 580, c["diffs"][:5]


@pytest.mark.parametrize("key", ["pe", "pe_veryfast"])
def test_golden_pe(eng, oracle, golden_oix, golden_dir, golden_ctxs, key):
    b1 = oracle.ReadBatch.from_fastq(os.path.join(golden_dir, "pe_1.fq"))
    b2 = oracle.ReadBatch.from_fastq(os.path.join(golden_dir, "pe_2.fq"))
    g1, g2, runs = golden_ctxs[key].map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    o1, o2, uo = oracle.map_pe(golden_oix, b1, b2, pe_method=5 if key.endswith("veryfast") else 4)
    assert_same(o1, uo, g1, runs)
    assert_same(o2, uo, g2, runs)
    sam = oracle.sam_header(golden_oix) + oracle.sam_pe(golden_oix, b1, b2, g1, g2, runs)
    c = synth.compare_sam(os.path.join(golden_dir, key + ".sam"), sam)
    assert c["identical"] == c["total"] == 860, c["diffs"][:5]


@pytest.fixture(scope="module")
def mid_env(eng, oracle, tmp_path_factory):
    """2 Mb repeat-rich reference indexed by the host builder."""
    d = tmp_path_factory.mktemp("mid")
    g = synth.make_genome(2_000_000, n_contigs=4, seed=77, repeat_frac=0.10, n_runs=[(2, 0.3, 1500)], tandem=20, segdup=4)
    fa, ufi = str(d / "ref.fa"), str(d / "ref.ufi")
    g.write_fasta(fa)
    make_ufi("mid_2mb_seed77", fa, ufi)
    return g, oracle.Index(ufi), eng.HostIndex(ufi)


@pytest.mark.parametrize("rl,sub,indel,method", [(150, 0.01, 0.001, 6), (150, 0.05, 0.01, 6), (250, 0.02, 0.002, 6),
                                                 (100, 0.03, 0.003, 7), (150, 0.05, 0.01, 7)])
def test_random_se(eng, oracle, mid_env, rl, sub, indel, method):
    g, oix, hix = mid_env
    reads, _ = synth.sim_se(g, 20000, rl, sub, indel, seed=rl + method)
    b = oracle.ReadBatch.from_arrays(reads)
    ctx = eng.Context(0, method=method)
    ctx.set_index(hix)
    res, runs = ctx.map_se(b.seqs, b.offs)
    ro, uo = oracle.map_se(oix, b, method=method, threads=os.cpu_count())
    assert_same(ro, uo, res, runs)
    ctx.close()


@pytest.mark.parametrize("rl,sub,indel,pe_method", [(150, 0.01, 0.001, 4), (150, 0.05, 0.01, 4), (250, 0.03, 0.003, 4),
                                                    (150, 0.03, 0.003, 5)])
def test_random_pe(eng, oracle, mid_env, rl, sub, indel, pe_method):
    g, oix, hix = mid_env
    r1, r2, _ = synth.sim_pe(g, 10000, rl, sub, indel, seed=rl + pe_method)
    r2 = r2.copy()
    r2[::50, : rl // 2] = r1[::50, : rl // 2]  # damage some mates so that ScanPair (mate rescue) fires
    b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
    ctx = eng.Context(0, pe_method=pe_method)
    ctx.set_index(hix)
    g1, g2, runs = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    o1, o2, uo, st = oracle.map_pe(oix, b1, b2, pe_method=pe_method, threads=os.cpu_count(), want_stats=True)
    if pe_method == 4:
        assert st["scan_calls"] > 0
    assert_same(o1, uo, g1, runs)
    assert_same(o2, uo, g2, runs)
    ctx.close()


def test_ragged_and_edge_reads(eng, oracle, mid_env):
    """Empty batch, reads shorter than the word length, ragged lengths 1..256, N / lower-case / IUPAC letters."""
    g, oix, hix = mid_env
    ctx = eng.Context(0)
    ctx.set_index(hix)
    res, runs = ctx.map_se(np.zeros(0, np.uint8), np.zeros(1, np.uint32))
    assert len(res) == 0
    rng = np.random.default_rng(3)
    lens = np.concatenate([[1, 5, 23, 24, 25, 47, 48, 96, 97, 255, 256], rng.integers(24, 257, size=3000)])
    seqs, offs = [], [0]
    for i, L in enumerate(lens):
        p = int(rng.integers(0, len(g.asc) - 300))
        s = g.asc[p:p + L].copy()
        if i % 7 == 0 and L > 40:
            s[rng.integers(0, L, size=3)] = ord("N")
        if i % 11 == 0:
            s = np.where((s >= 65) & (s <= 90), s + 32, s).astype(np.uint8)
        if i % 13 == 0 and L > 30:
            s[rng.integers(0, L)] = ord("R")
        if i % 17 == 0 and L > 30:
            s[rng.integers(0, L)] = ord("u")
        seqs.append(s)
        offs.append(offs[-1] + L)
    b = oracle.ReadBatch(np.concatenate(seqs), np.array(offs, dtype=np.uint32))
    # reads shorter than W make the reference underflow (SURVEY quirk 9); both sides report "no hit"
    res, runs = ctx.map_se(b.seqs, b.offs)
    ro, uo = oracle.map_se(oix, b, threads=4)
    assert_same(ro, uo, res, runs)
    # reads longer than URMB_MAX_READ_LEN are handled per read: reported unmapped with flag bit 6, the rest of the batch
    # is mapped exactly as without them (single-end and paired: the mate of an over-long read is not searched either)
    L0 = int(offs[40])
    long_read = g.asc[1000:1300].copy()
    mixed = np.concatenate([b.seqs[:L0], long_read, b.seqs[L0:]])
    moffs = np.concatenate([offs[:41], np.array(offs[40:]) + 300]).astype(np.uint32)
    r2_, u2_ = ctx.map_se(mixed, moffs)
    assert r2_[40]["flags"] == 0x40 and r2_[40]["db_pos"] == 0xFFFFFFFF and r2_[40]["mapq"] == 0
    assert canon(np.delete(r2_, 40), u2_) == canon(res, runs)
    assert ctx.unsupported_count() == (1, 1) and ctx.overflow_count()[1] == 0
    pr1, pr2, pu = ctx.map_pe(mixed, moffs, np.concatenate([b.seqs[:L0], b.seqs[:50], b.seqs[L0:]]),
                              np.concatenate([offs[:41], np.array(offs[40:]) + 50]).astype(np.uint32))
    assert pr1[40]["flags"] == 0x40 and pr2[40]["flags"] == 0x40 and ctx.unsupported_count() == (2, 3)
    q1, q2, qu = ctx.map_pe(b.seqs, b.offs, b.seqs, b.offs)
    assert canon(np.delete(pr1, 40), pu) == canon(q1, qu) and canon(np.delete(pr2, 40), pu) == canon(q2, qu)
    ctx.close()


def test_size_independent_properties(eng, oracle, mid_env):
    """Properties that also hold at BASELINE sizes: idempotence, batch-split invariance, permutation equivariance,
    and agreement of the pipelined (3-slot) interface with the synchronous one."""
    g, oix, hix = mid_env
    ctx = eng.Context(0)
    ctx.set_index(hix)
    r1, r2, _ = synth.sim_pe(g, 30000, 150, 0.02, 0.002, seed=5)
    b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
    a1, a2, ua = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    c1, c2, uc = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    full1, full2 = canon(a1, ua), canon(a2, ua)
    assert full1 == canon(c1, uc) and full2 == canon(c2, uc)
    # split into three slots, submitted back to back, waited afterwards
    n = b1.n
    cuts = [0, n // 3, 2 * n // 3, n]
    parts = []
    for k in range(3):
        lo, hi = cuts[k], cuts[k + 1]
        o = (b1.offs[lo:hi + 1] - b1.offs[lo]).astype(np.uint32)
        parts.append((np.ascontiguousarray(b1.seqs[b1.offs[lo]:b1.offs[hi]]), o,
                      np.ascontiguousarray(b2.seqs[b2.offs[lo]:b2.offs[hi]]), (b2.offs[lo:hi + 1] - b2.offs[lo]).astype(np.uint32)))
        ctx.submit(k, *parts[-1])
    got1, got2 = [], []
    for k in range(3):
        x1, x2, ux = ctx.wait(k, cuts[k + 1] - cuts[k], True)
        got1 += canon(x1, ux)
        got2 += canon(x2, ux)
    assert got1 == full1 and got2 == full2
    # permutation
    perm = np.random.default_rng(1).permutation(n)
    p1, p2 = oracle.ReadBatch.from_arrays(r1[perm]), oracle.ReadBatch.from_arrays(r2[perm])
    q1, q2, uq = ctx.map_pe(p1.seqs, p1.offs, p2.seqs, p2.offs)
    assert canon(q1, uq) == [full1[i] for i in perm]
    assert ctx.launch_count() >= 2 * 6
    ctx.close()


def _ctx_with_env(eng, hix, env, **kw):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        c = eng.Context(0, **kw)   # tuning variables are read at context creation
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    c.set_index(hix)
    return c


def test_chunk_size_invariance(eng, oracle, mid_env):
    """The staged search hands per-mate state over between small kernels chunk by chunk: results must not depend on the
    chunk size, on where the chunk borders fall, or on which stream the mate-rescue kernel runs (SE and PE)."""
    g, oix, hix = mid_env
    r1, r2, _ = synth.sim_pe(g, 6000, 150, 0.03, 0.003, seed=9)
    b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
    o1, o2, uo = oracle.map_pe(oix, b1, b2, threads=os.cpu_count())
    s1, us = oracle.map_se(oix, b1, threads=os.cpu_count())
    for env in ({"URMB_CHUNK_PAIRS": "1"}, {"URMB_CHUNK_PAIRS": "997"}, {"URMB_CHUNK_PAIRS": "5000", "URMB_RESCUE_INLINE": "1"},
                {"URMB_RESCUE_WARPS": "4"}):
        ctx = _ctx_with_env(eng, hix, env)
        if env.get("URMB_CHUNK_PAIRS") == "1":   # one pair per chunk: a small prefix is enough
            n = 150
            sb1 = oracle.ReadBatch(b1.seqs[:b1.offs[n]], b1.offs[:n + 1])
            sb2 = oracle.ReadBatch(b2.seqs[:b2.offs[n]], b2.offs[:n + 1])
            g1, g2, ug = ctx.map_pe(sb1.seqs, sb1.offs, sb2.seqs, sb2.offs)
            assert canon(g1, ug) == canon(o1[:n], uo) and canon(g2, ug) == canon(o2[:n], uo)
            x1, ux = ctx.map_se(sb1.seqs, sb1.offs)
            assert canon(x1, ux) == canon(s1[:n], us)
        else:
            g1, g2, ug = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
            assert_same(np.concatenate([o1, o2]), uo, np.concatenate([g1, g2]), ug)
            x1, ux = ctx.map_se(b1.seqs, b1.offs)
            assert_same(s1, us, x1, ux)
        ctx.close()


def test_dense_index_long_links(eng, oracle, tmp_path):
    """Mapping parity on an index full of long links (tallies 125 / 253, ufindex.cpp:256-300, 905-926): the host
    builder indexes the 2 Mb repeat-rich genome at load factor 0.95 (tens of thousands of long-link records); single-end
    (rows of both row kernels walk them) and paired-end results equal the oracle's on the same index."""
    g = synth.make_genome(2_000_000, n_contigs=4, seed=77, repeat_frac=0.10, n_runs=[(2, 0.3, 1500)], tandem=20, segdup=4)
    fa, ufi = str(tmp_path / "ref.fa"), str(tmp_path / "dense.ufi")
    g.write_fasta(fa)
    make_ufi("mid_2mb_seed77_load_factor_0.95", fa, ufi, ["-load_factor", "0.95"])
    oix, hix = oracle.Index(ufi), eng.HostIndex(ufi)
    tallies = oix.blob()[0::5]
    assert int(((tallies == 125) | (tallies == 253)).sum()) > 10000
    ctx = eng.Context(0)
    ctx.set_index(hix)
    reads, _ = synth.sim_se(g, 20000, 150, 0.02, 0.002, seed=31)
    b = oracle.ReadBatch.from_arrays(reads)
    res, runs = ctx.map_se(b.seqs, b.offs)
    ro, uo, st = oracle.map_se(oix, b, threads=os.cpu_count(), want_stats=True)
    assert st["row_hops"] > 100000
    assert_same(ro, uo, res, runs)
    r1, r2, _ = synth.sim_pe(g, 10000, 150, 0.02, 0.002, seed=32)
    b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
    g1, g2, ug = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    o1, o2, uo2 = oracle.map_pe(oix, b1, b2, threads=os.cpu_count())
    assert_same(np.concatenate([o1, o2]), uo2, np.concatenate([g1, g2]), ug)
    ctx.close()


def test_maxix_above_32(eng, oracle, tmp_path):
    """An index built with -maxix 100 (ufindexio.cpp:135-136) by the drop-in's GPU builder: byte-identical to the host
    builder's (and so to the reference's), and rows of 33 .. 100 positions (tandem arrays) are mapped as the oracle maps
    them, single-end and paired."""
    import subprocess
    g = synth.make_genome(1_000_000, n_contigs=3, seed=78, repeat_frac=0.30, n_runs=[(0, 0.3, 300)], tandem=40)
    fa, ufi, mine = str(tmp_path / "m.fa"), str(tmp_path / "m.ufi"), str(tmp_path / "mine.ufi")
    g.write_fasta(fa)
    make_ufi("m_1mb_seed78_maxix_100", fa, ufi, ["-maxix", "100"])
    r = subprocess.run([CLI, "-make_ufi", fa, "-output", mine, "-maxix", "100", "-gpu_build", "-quiet"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert open(mine, "rb").read() == open(ufi, "rb").read()
    oix, hix = oracle.Index(ufi), eng.HostIndex(mine)
    assert oix.max_ix == 100
    ctx = eng.Context(0)
    ctx.set_index(hix)
    reads, _ = synth.sim_se(g, 20000, 150, 0.02, 0.002, seed=31)
    b = oracle.ReadBatch.from_arrays(reads)
    res, runs = ctx.map_se(b.seqs, b.offs)
    ro, uo, st = oracle.map_se(oix, b, threads=os.cpu_count(), want_stats=True)
    assert st["row_hops_long"] > 20 * b.n
    assert_same(ro, uo, res, runs)
    r1, r2, _ = synth.sim_pe(g, 10000, 250, 0.02, 0.002, seed=32)
    b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
    g1, g2, ug = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    o1, o2, uo2 = oracle.map_pe(oix, b1, b2, threads=os.cpu_count())
    assert_same(np.concatenate([o1, o2]), uo2, np.concatenate([g1, g2]), ug)
    ctx.close()


def test_first_look(eng, oracle, mid_env):
    """The probe kernel's first look (paired input): the pairs it finishes -- the seed-loop exit of Search4/5,
    search2m4.cpp:79-142, 203-205 -- carry the oracle's records, a third of clean pairs take it, and switching it off
    (URMB_FLAGS bit 9) changes nothing.  Also -map2 -veryfast (Search5), 250-base reads and reads shorter than a word."""
    g, oix, hix = mid_env
    for rl, sub, indel, pm in ((150, 0.01, 0.001, 4), (150, 0.01, 0.001, 5), (250, 0.005, 0.0005, 4), (100, 0.0, 0.0, 4)):
        r1, r2, _ = synth.sim_pe(g, 8000, rl, sub, indel, seed=41 + rl)
        b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
        o1, o2, uo = oracle.map_pe(oix, b1, b2, pe_method=pm, band_radius=4 if pm == 5 else -1, threads=os.cpu_count())
        got = []
        for env in ({}, {"URMB_FLAGS": "512"}):
            ctx = _ctx_with_env(eng, hix, env, pe_method=pm, band_radius=4 if pm == 5 else -1)
            g1, g2, ug = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
            assert_same(np.concatenate([o1, o2]), uo, np.concatenate([g1, g2]), ug)
            got.append(ctx.first_look_count()[0])
            ctx.close()
        assert got[1] == 0 and got[0] > 0.2 * b1.n, got
    # ragged pairs: a mate shorter than a word, an empty mate, invalid letters -- never finished by the first look wrongly
    r1, r2, _ = synth.sim_pe(g, 64, 150, 0.0, 0.0, seed=5)
    rows1 = [bytes(r) for r in r1]
    rows2 = [bytes(r) for r in r2]
    rows1[0], rows2[1], rows1[2], rows2[3] = rows1[0][:20], b"", rows1[2][:30], b"N" * 150
    rows1[4] = rows1[4][:70] + b"N" + rows1[4][71:]
    rows2[5] = rows2[5].lower()
    def batch(rows):
        return oracle.ReadBatch(np.frombuffer(b"".join(rows), dtype=np.uint8), np.concatenate([[0], np.cumsum([len(x) for x in rows])]).astype(np.uint32))

    b1, b2 = batch(rows1), batch(rows2)
    o1, o2, uo = oracle.map_pe(oix, b1, b2, threads=2)
    ctx = eng.Context(0)
    ctx.set_index(hix)
    g1, g2, ug = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
    assert_same(np.concatenate([o1, o2]), uo, np.concatenate([g1, g2]), ug)
    ctx.close()


def test_big_capacity_rerun_and_legacy_rescue(eng, oracle, mid_env):
    """Reads that overflow a per-mate capacity are mapped again by the kernels compiled with big capacities (urmb_big.cu),
    in stream behind the mate rescue (URMB_FLAGS bit 8 forces it for every fifth read) or, for what is left, from the host
    in urmb_wait (URMB_FORCE_RERUN forces it for every third unit): the results must not change (SE and PE, path runs and
    second hits included).
    The legacy mate-rescue kernel (no rescue pool) and the rescue in rounds of window scans and batched full-window DPs
    (URMB_RESCUE_ROUNDS; the default runs the DPs in place) must agree as well."""
    g, oix, hix = mid_env
    r1, r2, _ = synth.sim_pe(g, 5000, 150, 0.04, 0.006, seed=21)
    r2 = r2.copy()
    r2[::20, :75] = r1[::20, :75]   # damaged mates: mate rescue
    b1, b2 = oracle.ReadBatch.from_arrays(r1), oracle.ReadBatch.from_arrays(r2)
    o1, o2, uo = oracle.map_pe(oix, b1, b2, threads=os.cpu_count())
    s1, us = oracle.map_se(oix, b1, threads=os.cpu_count())
    for env in ({"URMB_FORCE_RERUN": "3"}, {"URMB_FLAGS": "256"}, {"URMB_FLAGS": "256", "URMB_RESCUE_INLINE": "1"},
                {"URMB_RESCUE_LEGACY": "1"}, {"URMB_RESCUE_ROUNDS": "2"}, {"URMB_RESCUE_ROUNDS": "6"}):
        ctx = _ctx_with_env(eng, hix, env, want_second=True)
        g1, g2, ug = ctx.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
        assert_same(np.concatenate([o1, o2]), uo, np.concatenate([g1, g2]), ug)
        sec = [x.copy() for x in ctx.second_hits(0, b1.n)]
        x1, ux = ctx.map_se(b1.seqs, b1.offs)
        assert_same(s1, us, x1, ux)
        assert ctx.overflow_count()[1] == 0
        ctx.close()
        ref = eng.Context(0, want_second=True)
        ref.set_index(hix)
        ref.map_pe(b1.seqs, b1.offs, b2.seqs, b2.offs)
        rs = ref.second_hits(0, b1.n)
        assert (sec[0] == rs[0]).all() and (sec[1] == rs[1]).all()
        ref.close()


def test_human_scale_properties(eng):
    """BASELINE.json's full-size index (3.1 Gb reference, 27 GB table, built on the GPU) with properties that need no
    oracle: reads map back to where they were drawn from, results are idempotent, independent of the chunk size and of
    how a batch is split over the three pipeline slots.  (bench.py additionally compares 2 M SAM records with the
    reference binary at this size.)"""
    import torch
    from urmap_b200 import gpu_synth, index_build
    free, _ = torch.cuda.mem_get_info()
    if free < 60e9:
        pytest.skip("needs 60 GB of free HBM")
    dev = torch.device("cuda", 0)
    seq, names, lens, offsets, sds = gpu_synth.make_seqdata(3_100_000_000, dev, n_contigs=24, human_ratios=True)
    slots = index_build.slot_count_for(names, lens)
    assert slots == 5392814809   # first prime >= FASTA bytes / 0.6 (SURVEY.md §8)
    blob = torch.empty(5 * slots + 16, dtype=torch.uint8, device=dev)
    st = index_build.build_index_device(seq.data_ptr(), sds, slots, blob.data_ptr())
    assert st["truncated"] == 0 and st["indexed"] > 2_900_000_000
    n, RL = 200_000, 150
    r1, r2, t1, t2, plus1 = gpu_synth.sim_pe(seq, lens, offsets, n, dev, RL, 0.01, 0.001, seed=4242, return_truth=True)
    a1, a2 = r1.cpu().numpy().reshape(-1), r2.cpu().numpy().reshape(-1)
    t1, t2, plus1 = t1.cpu().numpy(), t2.cpu().numpy(), plus1.cpu().numpy()
    offs = (np.arange(n + 1, dtype=np.uint32) * RL)
    desc = (24, 32, sds, slots, blob.data_ptr(), seq.data_ptr())

    def run(env, split=None):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            ctx = eng.Context(0)
        finally:
            for k, v in old.items():
                os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
        ctx.attach_index(*desc, keepalive=(seq, blob))
        if split is None:
            x1, x2, ux = ctx.map_pe(a1, offs, a2, offs)
            out = canon(x1, ux), canon(x2, ux), x1.copy(), x2.copy()
        else:
            cuts = [0, split, 2 * split, n]
            for k in range(3):
                lo, hi = cuts[k], cuts[k + 1]
                o = (np.arange(hi - lo + 1, dtype=np.uint32) * RL)
                ctx.submit(k, a1[lo * RL:hi * RL], o, a2[lo * RL:hi * RL], o)
            c1, c2 = [], []
            for k in range(3):
                x1, x2, ux = ctx.wait(k, cuts[k + 1] - cuts[k], True)
                c1 += canon(x1, ux)
                c2 += canon(x2, ux)
            out = c1, c2, None, None
        ctx.close()
        return out

    f1, f2, x1, x2 = run({})
    # truth: confidently mapped mates sit where they were drawn from (alignment start within the read's own indels)
    for x, t, plus in ((x1, t1, plus1), (x2, t2, ~plus1)):
        conf = x["mapq"] >= 20
        assert conf.mean() > 0.8, float(conf.mean())
        ok = (np.abs(x["db_pos"].astype(np.int64) - t) <= 12) & (((x["flags"] & 1) != 0) == plus)
        assert ok[conf].mean() > 0.999, float(ok[conf].mean())
    g1, g2, _, _ = run({"URMB_CHUNK_PAIRS": "30011"})
    assert g1 == f1 and g2 == f2
    h1, h2, _, _ = run({}, split=70_001)
    assert h1 == f1 and h2 == f2
    del blob, seq
    torch.cuda.empty_cache()
