"""The device index builder (urmb_build.cu) must produce the reference's UFI blob byte for byte (segments cut by a max-plus
carry scan, the reference's insertions replayed in genome order inside each segment, long links included); only a table
whose lists would have to be truncated must be reported instead."""
import os
import struct
import sys

import numpy as np
import pytest

from conftest import CLI, ROOT, have_gpu, make_ufi

sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))


def _swap_blob(src_ufi, blob, slot_count, out):
    raw = open(src_ufi, "rb").read()
    hdr = raw.index(struct.pack("<I", 0x55464932)) + 4
    open(out, "wb").write(raw[:hdr] + blob.tobytes() + raw[hdr + 5 * slot_count:])


def test_prime_and_fasta_size(oracle, golden_dir):
    from urmap_b200 import index_build
    for n in (100, 101, 5000, int(5083340 / 0.6), int(3151666838 / 0.6)):
        assert index_build.get_prime(n) == oracle.get_prime(n)
    names, lens = ["ctg1", "ctg2", "ctg3"], [50000, 50000, 50000]
    assert index_build.fasta_bytes(names, lens) == os.path.getsize(os.path.join(golden_dir, "ref.fa"))


def test_emulated_builder_matches_reference(oracle, golden_oix, golden_dir, tmp_path):
    import emu_py
    blob, stats = emu_py.emu_build_index(golden_oix.seq(), golden_oix.slot_count, golden_oix.word_length, golden_oix.max_ix)
    assert stats[1] == 0 and stats[2] == 0
    out = str(tmp_path / "emu.ufi")
    _swap_blob(os.path.join(golden_dir, "ref.ufi"), blob, golden_oix.slot_count, out)
    assert np.array_equal(blob, np.asarray(golden_oix.blob()[:5 * golden_oix.slot_count]))   # byte-identical
    mine = oracle.Index(out)
    assert oracle.index_functional_diff(golden_oix, mine)[0] == 0
    if os.path.exists(oracle.REF_BIN):  # the reference's own validator accepts it (ufistats.cpp:141)
        oracle.run_reference(["-ufi_validate", out])


@pytest.mark.parametrize("extra,long_links", [([], False), (["-veryfast"], False), (["-maxix", "5", "-wordlength", "20"], False),
                                              (["-maxix", "100"], True),
                                              (["-load_factor", "0.8"], True), (["-load_factor", "0.95"], True)])
def test_emulated_builder_options(oracle, built_lib, tmp_path, extra, long_links):
    """Repeat-rich 400 kb genome under the reference's index options: byte-identical to the reference's file (stored digest),
    including the dense tables in which the reference needs long links (two slots per element: the repair pass replays
    those segments)."""
    import emu_py
    from urmap_b200 import synth
    g = synth.make_genome(400_000, n_contigs=3, seed=31, repeat_frac=0.15, n_runs=[(1, 0.3, 900)], tandem=15, segdup=4)
    fa, ufi = str(tmp_path / "r.fa"), str(tmp_path / "r.ufi")
    g.write_fasta(fa)
    make_ufi("r_400kb_seed31" + "".join("_" + e.lstrip("-") for e in extra), fa, ufi, extra)
    ref = oracle.Index(ufi)
    blob, stats = emu_py.emu_build_index(ref.seq(), ref.slot_count, ref.word_length, ref.max_ix)
    want = np.asarray(ref.blob()[:5 * ref.slot_count])
    tl = want[0::5]
    assert (int(((tl == 125) | (tl == 253)).sum()) > 0) == long_links   # the case is what it claims to be
    assert stats[1] == 0 and np.array_equal(blob, want)


@pytest.mark.gpu
def test_gpu_builder_matches_reference(oracle, built_lib, tmp_path):
    if not have_gpu():
        pytest.skip("no CUDA device")
    import subprocess
    import torch
    from urmap_b200 import index_build, synth
    g = synth.make_genome(3_000_000, n_contigs=5, seed=9, repeat_frac=0.15, n_runs=[(1, 0.2, 4000)], tandem=30, segdup=5)
    fa, ufi = str(tmp_path / "r.fa"), str(tmp_path / "r.ufi")
    g.write_fasta(fa)
    make_ufi("r_3mb_seed9", fa, ufi)
    ref = oracle.Index(ufi)
    assert index_build.slot_count_for(g.names, g.lens) == ref.slot_count
    seq = torch.from_numpy(np.concatenate([ref.seq(), np.zeros(4096, np.uint8)])).cuda()
    blob = torch.empty(5 * ref.slot_count + 16, dtype=torch.uint8, device="cuda")
    st = index_build.build_index_device(seq.data_ptr(), ref.seq_size, ref.slot_count, blob.data_ptr())
    assert st["truncated"] == 0
    out = str(tmp_path / "gpu.ufi")
    mine_blob = blob[:5 * ref.slot_count].cpu().numpy()
    assert np.array_equal(mine_blob, np.asarray(ref.blob()[:5 * ref.slot_count]))   # byte-identical to the reference
    _swap_blob(ufi, mine_blob, ref.slot_count, out)
    assert open(out, "rb").read() == open(ufi, "rb").read()
    mine = oracle.Index(out)
    assert oracle.index_functional_diff(ref, mine)[0] == 0
    r = subprocess.run([CLI, "-ufi_validate", out, "-quiet"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    if os.path.exists(oracle.REF_BIN):   # the reference's own validator accepts it (ufistats.cpp:141)
        oracle.run_reference(["-ufi_validate", out])
    # and the engine maps identically with either index
    from urmap_b200 import engine
    reads, _ = synth.sim_se(g, 5000, 150, 0.03, 0.003, seed=4)
    b = oracle.ReadBatch.from_arrays(reads)
    res = []
    for path in (ufi, out):
        ctx = engine.Context(0)
        ctx.set_index(engine.HostIndex(path))
        r, u = ctx.map_se(b.seqs, b.offs)
        res.append([tuple(int(x[f]) for f in ("db_pos", "score", "best", "second", "mapq", "flags")) for x in r])
        ctx.close()
    assert res[0] == res[1]
