// tests/emu/emu_fasta.cpp -- DEBUGGING HARNESS, NOT PRODUCT CODE (see tests/emu/cuda_runtime.h).
// The FASTA parse kernels of urmap_b200/csrc/urmb_fasta.cu on the lock-step warp emulator of emu.cpp (libemu_fasta.so,
// built by emu_fasta_py.py).
#include "emu.cpp"   // the emulator (and the kernels it compiles)
#include "../../urmap_b200/csrc/urmb_fasta.cu"

// FASTA parse kernels (urmb_fasta.cu) under emulation, in the order fasta_parse_device launches them.  The results stay here
// until the next call: emu_fasta_seq / emu_fasta_record / emu_fasta_dropped / emu_fasta_error read them.
static std::vector<uint8_t> g_fa_seq;
static FastaTable g_fa_tab;
static std::string g_fa_err;
extern "C" int emu_parse_fasta(const uint8_t *fa_in, uint64_t len) {
    g_fa_seq.clear();
    g_fa_tab = FastaTable();
    g_fa_err.clear();
    std::vector<uint8_t> fa(fasta_padded_len(len), 0);
    if (len) memcpy(fa.data(), fa_in, len);
    FastaArgs a{};
    a.fa = fa.data();
    a.len = len;
    a.ntiles = fasta_tiles(len);
    std::vector<uint32_t> tcount(a.ntiles + 1);
    std::vector<uint64_t> tscan(a.ntiles + 1);
    a.tcount = tcount.data();
    a.tscan = tscan.data();
    const int blocks = (int)((a.ntiles + kFaWarps - 1) / kFaWarps);
    if (a.ntiles) emu::launch([&]() { fa_hdr_kernel<false>(a); }, blocks, 32 * kFaWarps, 0);
    emu::launch([&]() { fa_scan_kernel(a.tcount, a.tscan, a.ntiles); }, 1, 32, 0);
    a.nrec = tscan[a.ntiles];
    std::vector<uint64_t> h(a.nrec + 1), e(a.nrec + 1), hk(a.nrec + 1);
    a.h = h.data();
    a.e = e.data();
    a.hk = hk.data();
    auto grid = [](uint64_t n) { return (int)(n / 256 + 1); };
    if (a.ntiles) emu::launch([&]() { fa_hdr_kernel<true>(a); }, blocks, 32 * kFaWarps, 0);
    emu::launch([&]() { fa_hdr_end_kernel(a); }, grid(a.nrec), 256, 0);
    if (a.ntiles) emu::launch([&]() { fa_count_kernel(a); }, blocks, 32 * kFaWarps, 0);
    emu::launch([&]() { fa_scan_kernel(a.tcount, a.tscan, a.ntiles); }, 1, 32, 0);
    emu::launch([&]() { fa_rec_kernel(a); }, grid(a.nrec), 256, 0);
    g_fa_err = fasta_check_head(fa.data(), h[0]);
    if (!g_fa_err.empty()) return URMB_E_IO;
    g_fa_err = fasta_table(fa.data(), h.data(), e.data(), hk.data(), a.nrec, g_fa_tab);
    if (!g_fa_err.empty()) return URMB_E_UNSUPPORTED;
    a.nkept_rec = g_fa_tab.nstart.size();
    a.nstart = g_fa_tab.nstart.data();
    g_fa_seq.assign(g_fa_tab.seq_size + URMB_SEQ_PAD, 0xEE);
    memset(g_fa_seq.data() + g_fa_tab.seq_size, 0, URMB_SEQ_PAD);
    a.out = g_fa_seq.data();
    if (a.ntiles) emu::launch([&]() { fa_scatter_kernel(a); }, blocks, 32 * kFaWarps, 0);
    emu::launch([&]() { fa_pad_kernel(a); }, grid(a.nkept_rec), 256, 0);
    return 0;
}
extern "C" uint64_t emu_fasta_seq(const uint8_t **p) { *p = g_fa_seq.data(); return g_fa_seq.size(); }
extern "C" uint32_t emu_fasta_n_records() { return (uint32_t)g_fa_tab.labels.size(); }
extern "C" const char *emu_fasta_record(uint32_t i, uint32_t *label_len, uint32_t *length, uint32_t *offset) {
    *label_len = (uint32_t)g_fa_tab.labels[i].size();
    *length = g_fa_tab.lengths[i];
    *offset = g_fa_tab.offsets[i];
    return g_fa_tab.labels[i].data();
}
extern "C" uint32_t emu_fasta_n_dropped() { return (uint32_t)g_fa_tab.dropped.size(); }
extern "C" const char *emu_fasta_dropped(uint32_t i, uint32_t *label_len) {
    *label_len = (uint32_t)g_fa_tab.dropped[i].size();
    return g_fa_tab.dropped[i].data();
}
extern "C" const char *emu_fasta_error() { return g_fa_err.c_str(); }
