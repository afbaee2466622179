// CPU thread-emulator for the block encoder in 7bgzf_b200/csrc/bgzf_block.h.
// TEST/DEVELOPMENT INFRASTRUCTURE: it runs the very phase functions the CUDA kernel runs, one "thread" at a
// time, so the algorithm can be checked (and race-checked, by permuting the thread order) without a GPU.
// The product never links this.
//
//   emul compress <level> <in> <out.bgz> [order]   order: 0 forward, 1 reverse, 2 shuffled
//   library: int bgemul_compress_block(const uint8_t* src, uint32_t n, int level, int order, uint8_t* dst /*65536*/, uint32_t* dlen)
//            void bgemul_last_trees(uint32_t out[7]), bgemul_last_ties(uint32_t out[4])   the Huffman trees of the last block (see below)
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>
#include "../../7bgzf_b200/csrc/bgzf_block.h"
#include "../../7bgzf_b200/csrc/bgzf_tables.h"

namespace {
struct Emu {
    std::vector<uint32_t> dataw, regA, regB, R, out, crcpow, cand;
    uint8_t litflag[256];
    uint32_t crctab[256];
    uint32_t scal[BG_S_COUNT];
    Emu() : dataw(BG_DATA_BYTES / 4), regA(131072 / 4), regB(32768 / 4), R(BG_MAX_BLOCK + 8), out(BG_SLOT_BYTES / 4), crcpow(BG_THREADS), cand(4 * BG_MAX_BLOCK)
    {
        bg_make_crc_table(crctab);
        bg_make_crc_pow(crcpow.data(), BG_THREADS);
    }
};

typedef void (*phase_fn)(const BgCtx &, uint32_t, uint32_t);

void run(phase_fn f, const BgCtx &c, int order, uint32_t seed)
{
    const uint32_t T = BG_THREADS;
    std::vector<uint32_t> idx(T);
    std::iota(idx.begin(), idx.end(), 0u);
    if (order == 1) std::reverse(idx.begin(), idx.end());
    if (order == 2) {
        uint32_t s = seed * 2654435761u + 12345u;
        for (uint32_t i = T - 1; i > 0; i--) { s = s * 1664525u + 1013904223u; std::swap(idx[i], idx[(s >> 8) % (i + 1)]); }
    }
    for (uint32_t t : idx) f(c, t, T);
}

/* the tree over the m ascending keys (m <= 32), built by the kernel's merge on copies: out[0] = the overflow the code-length
 * repair of bg_huff_lengths() starts from (nodes deeper than maxbits), out[1] = leaves of the same weight as the leaf
 * before them, out[2] = picks of the merge where the lightest leaf and the lightest merged node weigh the same (the leaf
 * goes first) */
void tree_stats(const uint32_t *keys, uint32_t m, uint32_t maxbits, uint32_t out[3])
{
    out[0] = out[1] = out[2] = 0;
    if (m < 2) return;
    uint32_t w[64];
    uint16_t par[64];
    for (uint32_t i = 0; i < m; i++) w[i] = keys[i] >> 9;
    bg_huff_merge(m, w, par);
    const uint32_t root = 2 * m - 2;
    for (uint32_t i = 0; i < root; i++) {
        uint32_t d = 0;
        for (uint32_t x = i; x != root; x = par[x]) d++;
        out[0] += d > maxbits;
    }
    for (uint32_t i = 1; i < m; i++) out[1] += w[i] == w[i - 1];
    for (uint32_t a = 0, b = m, e = m; e < 2 * m - 1; e++)     /* the picks again, from the weights the merge left */
        for (int k = 0; k < 2; k++) {
            if (a < m && b < e && w[a] == w[b]) out[2]++;
            if (a < m && (b >= e || w[a] <= w[b])) a++; else b++;
        }
}
}  // namespace

/* statistics of the trees of the last bgemul_compress_block call's final pass (the one it emits):
 * BTYPE, then used symbols and overflow (nodes deeper than the length limit) of the litlen, distance and precode codes */
static uint32_t g_emul_trees[7];
extern "C" void bgemul_last_trees(uint32_t out[7]) { memcpy(out, g_emul_trees, sizeof g_emul_trees); }
/* ties of the same call's distance and precode trees: equal leaf weights, then leaf / merged-node ties, of each (tree_stats) */
static uint32_t g_emul_ties[4];
extern "C" void bgemul_last_ties(uint32_t out[4]) { memcpy(out, g_emul_ties, sizeof g_emul_ties); }

static uint32_t g_emul_hdr = 18;
/* member framing of the following bgemul_compress_block calls: 18 = BGZF (default), 20 = MiGz */
extern "C" void bgemul_set_header_bytes(uint32_t hdr) { g_emul_hdr = hdr == 20 ? 20 : 18; }
/* piece mode of the following calls (BgCtx.piece): head / tail gap bytes and whether the piece is the final DEFLATE block;
 * enable = 0 returns to members */
static uint32_t g_emul_piece = 0, g_emul_head = 0, g_emul_tail = 0, g_emul_final = 1, g_emul_crc = 0;
extern "C" void bgemul_set_piece(uint32_t enable, uint32_t head_gap, uint32_t tail_gap, uint32_t final)
{
    g_emul_piece = enable ? 1 : 0;
    g_emul_head = head_gap;
    g_emul_tail = tail_gap;
    g_emul_final = final ? 1 : 0;
}
extern "C" uint32_t bgemul_last_crc(void) { return g_emul_crc; }
/* piece mode: the first `hist` bytes of the following calls' src are history (a multiple of 272, at most 32640) */
static uint32_t g_emul_hist = 0;
extern "C" void bgemul_set_history(uint32_t hist) { g_emul_hist = hist; }

extern "C" int bgemul_compress_block(const uint8_t *src, uint32_t n, int level, int order, uint8_t *dst, uint32_t *dlen)
{
    static Emu *e = new Emu();
    if (n > BG_MAX_BLOCK) return -1;
    // poison what the kernel would find uninitialised
    std::fill(e->regA.begin(), e->regA.end(), 0xA5A5A5A5u);
    std::fill(e->regB.begin(), e->regB.end(), 0x5A5A5A5Au);
    std::fill(e->R.begin(), e->R.end(), 0xDEADBEEFu);
    std::fill(e->out.begin(), e->out.end(), 0xFFFFFFFFu);
    std::fill(e->dataw.begin(), e->dataw.end(), 0xEEEEEEEEu);
    memcpy(e->dataw.data(), src, n);
    BgCtx c;
    c.dataw = e->dataw.data();
    c.prev = (uint16_t *)e->regA.data();
    c.stepcode = (uint8_t *)e->regA.data();
    c.jump8 = c.stepcode + 65536;
    c.offarr = (uint16_t *)c.jump8;
    c.head = (uint16_t *)e->regB.data();
    c.regb = (uint8_t *)e->regB.data();
    c.litflag = e->litflag;
    c.crctab = e->crctab;
    c.scal = e->scal;
    c.R = e->R.data();
    c.cand = e->cand.data();
    c.out = e->out.data();
    c.crcpow = e->crcpow.data();
    c.perm = nullptr;
    c.n = n;
    if (g_emul_hist % BG_HISTORY_STEP || g_emul_hist > BG_MAX_HISTORY || g_emul_hist > n) return -3;
    c.frame = g_emul_piece ? bg_frame(g_emul_head, g_emul_tail, g_emul_final, 1u, g_emul_hist) : bg_frame(g_emul_hdr, 8u, 1u, 0u);
    c.prm = bg_level_params(level);
    memset(g_emul_trees, 0, sizeof g_emul_trees);
    memset(g_emul_ties, 0, sizeof g_emul_ties);
    uint32_t k = 0;
    run(bg_phase_init, c, order, k++);
    run(bg_phase_scan, c, order, k++);
    run(bg_phase_count, c, order, k++);
    run(bg_phase_settle, c, order, k++);
    run(bg_phase_hash, c, order, k++);
    bg_build_sequential(c);
    run(bg_phase_search_clear, c, order, k++);
    run(bg_phase_search1, c, order, k++);
    if (c.scal[BG_S_DEPTH] > 1) {
        run([](const BgCtx &cc, uint32_t t, uint32_t T) { bg_phase_search_todo(cc, t, T, 0u, 1u); }, c, order, k++);
        run(bg_phase_search2, c, order, k++);
    }
    for (int pass = 0; pass <= c.prm.opt_passes; pass++) {
        if (pass == 0) {
            run(bg_phase_accept, c, order, k++);
        } else {
            run(bg_phase_costs, c, order, k++);
            // the rings live in the (dead) second half of region A, like in the kernel
            uint32_t *rings = (uint32_t *)(c.stepcode + 65536);
            for (uint32_t t = 0; t < BG_THREADS; t++) bg_phase_dp(c, order == 1 ? BG_THREADS - 1 - t : t, BG_THREADS, rings);
        }
        run(bg_phase_history_steps, c, order, k++);
        run(bg_phase_jump, c, order, k++);
        run(bg_phase_walk_clear, c, order, k++);
        run(bg_phase_walk_mark, c, order, k++);
        run(bg_phase_walk_list, c, order, k++);
        run(bg_phase_walk_a, c, order, k++);
        run(bg_phase_walk_b, c, order, k++);
        run(bg_phase_walk_c, c, order, k++);
        if (c.scal[BG_S_WALKEND] != n) { fprintf(stderr, "emul: walk ended at %u, n=%u\n", c.scal[BG_S_WALKEND], n); return -2; }
        run(bg_phase_clear_freq, c, order, k++);
        run(bg_phase_tally, c, order, k++);
        run(bg_phase_lkeys, c, order, k++);
        {   // twin of the kernel's bitonic sort
            uint32_t *keys = (uint32_t *)(c.regb + BG_B_KEYS);
            std::sort(keys, keys + 512);
        }
        run(bg_phase_huff_prep, c, order, k++);
        run(bg_phase_huff, c, order, k++);
        {
            uint32_t st[3];
            tree_stats((const uint32_t *)(c.regb + BG_B_DKEYS), c.scal[BG_S_DM], 15, st);
            g_emul_trees[3] = c.scal[BG_S_DM];
            g_emul_trees[4] = st[0];
            g_emul_ties[0] = st[1];
            g_emul_ties[1] = st[2];
        }
        run(bg_phase_huff_depth, c, order, k++);
        g_emul_trees[1] = c.scal[BG_S_HM];
        g_emul_trees[2] = c.scal[BG_S_HOVF];
        run(bg_phase_huff_fix, c, order, k++);
        run(bg_phase_huff_assign, c, order, k++);
    }
    run(bg_phase_hdr1, c, order, k++);
    run(bg_phase_hdr2, c, order, k++);
    run(bg_phase_hdr3, c, order, k++);
    uint32_t nitems = 0;
    {   // twin of the kernel's block-wide exclusive scan
        uint32_t *cb = (uint32_t *)(c.regb + BG_B_CBITS);
        for (uint32_t i = 0; i < BG_MAX_CHUNKS; i++) { uint32_t v = cb[i]; cb[i] = nitems; nitems += v; }
    }
    run(bg_phase_hdr4, c, order, k++);
    run(bg_phase_hdr4b, c, order, k++);
    {
        uint32_t st[3];
        tree_stats((const uint32_t *)(c.regb + BG_B_PKEYS), c.scal[BG_S_PM], 7, st);
        g_emul_trees[5] = c.scal[BG_S_PM];
        g_emul_trees[6] = st[0];
        g_emul_ties[2] = st[1];
        g_emul_ties[3] = st[2];
    }
    for (uint32_t t = 0; t < BG_THREADS; t++) bg_phase_hdr5(c, t, BG_THREADS, nitems);
    {   // cross-check against the sequential rule
        static uint16_t ref_items[400]; uint32_t ref_pf[19];
        uint32_t ni = bg_header_items(c.regb + BG_B_LLEN, c.scal[BG_S_NL], c.regb + BG_B_DLEN, c.scal[BG_S_ND], ref_items, ref_pf);
        if (ni != nitems || memcmp(ref_items, c.regb + BG_B_ITEMS, ni * 2) || memcmp(ref_pf, c.regb + BG_B_PFREQ, 19 * 4)) {
            fprintf(stderr, "emul: parallel header items differ from the sequential rule (%u vs %u)\n", nitems, ni);
            return -4;
        }
    }
    run(bg_phase_decide_b, c, order, k++);
    g_emul_trees[0] = c.scal[BG_S_BTYPE];
    run(bg_phase_codes_a, c, order, k++);
    run(bg_phase_codes_b, c, order, k++);
    run(bg_phase_codes_c, c, order, k++);
    run(bg_phase_tabs, c, order, k++);
    run(bg_phase_hdr_bits, c, order, k++);
    {   // twin of the kernel's block-wide exclusive scan
        uint32_t *io = (uint32_t *)(c.regb + BG_B_IOFF), acc = 0;
        for (uint32_t i = 0; i < BG_MAX_CHUNKS; i++) { uint32_t v = io[i]; io[i] = acc; acc += v; }
    }
    run(bg_phase_sizes, c, order, k++);
    {   // twin of the kernel's block-wide exclusive scan
        uint32_t *cb = (uint32_t *)(c.regb + BG_B_CBITS), acc = 0;
        for (uint32_t i = 0; i < BG_MAX_CHUNKS; i++) { uint32_t v = cb[i]; cb[i] = acc; acc += v; }
        if (c.scal[BG_S_BTYPE] && acc + ((uint8_t *)(c.regb + BG_B_LLEN))[256] != c.scal[BG_S_TOKBITS]) {
            fprintf(stderr, "emul: token bits %u + eob != %u\n", acc, c.scal[BG_S_TOKBITS]);
            return -3;
        }
    }
    if (c.scal[BG_S_STATUS]) return 1;
    run(bg_phase_zero_out, c, order, k++);
    run(bg_phase_emit, c, order, k++);
    uint32_t total = bg_f_hdr(c) + c.scal[BG_S_PAYLOAD] + bg_f_trl(c);
    g_emul_crc = c.scal[BG_S_CRC];
    memcpy(dst, e->out.data(), total);
    *dlen = total;
    return 0;
}

#ifdef EMUL_MAIN
int main(int argc, char **argv)
{
    if (argc < 5) { fprintf(stderr, "usage: emul compress <level> <in> <out> [order] [blocksize]\n"); return 2; }
    int level = atoi(argv[2]), order = argc > 5 ? atoi(argv[5]) : 0;
    uint32_t bs = argc > 6 ? (uint32_t)strtoul(argv[6], 0, 0) : 0xff00u;
    FILE *f = fopen(argv[3], "rb");
    if (!f) { perror(argv[3]); return 1; }
    std::vector<uint8_t> in;
    { uint8_t buf[65536]; size_t r; while ((r = fread(buf, 1, sizeof buf, f)) > 0) in.insert(in.end(), buf, buf + r); }
    fclose(f);
    FILE *o = fopen(argv[4], "wb");
    uint8_t dst[65536];
    size_t total = 0;
    for (size_t off = 0; off < in.size(); off += bs) {
        uint32_t n = (uint32_t)std::min<size_t>(bs, in.size() - off), dl = 0;
        int r = bgemul_compress_block(in.data() + off, n, level, order, dst, &dl);
        if (r) { fprintf(stderr, "block at %zu: error %d\n", off, r); return 1; }
        fwrite(dst, 1, dl, o);
        total += dl;
    }
    { uint32_t dl = 0; bgemul_compress_block(in.data(), 0, level, order, dst, &dl); fwrite(dst, 1, dl, o); total += dl; }
    fclose(o);
    fprintf(stderr, "in=%zu out=%zu ratio=%.4f\n", in.size(), total, in.size() ? (double)total / in.size() : 0.0);
#ifdef BG_STATS
    fprintf(stderr, "search steps/position %.2f (tail checks %.2f)\n", (double)bg_stat_steps / in.size(), (double)bg_stat_tail / in.size());
#endif
    return 0;
}
#endif
