/*
 * containers.c — the other block-gzip containers of the reference's applet family and whole-stream gzip, written around
 * the raw DEFLATE pieces the compress kernel makes in piece mode (SURVEY 8f ranks 3 and 4).  Only the framing differs
 * from BGZF; what each container looks like follows the reference's writers:
 *   MiGz     applet/7migz.c:133-243       gzip subfield "MZ" (u32 DEFLATE size), members of N KiB
 *   GZinga   applet/7gzinga.c:78-216      members with an empty comment + an index member ("n:end;" list in its comment)
 *   dictzip  applet/7dictzip.c:177-318    subfield "RA" (version, chunk length, chunk count, u16 sizes), full-flushed chunks,
 *                                         an empty static block, CRC32, ISIZE; members of at most 32762 chunks
 *   RAZF     applet/7razf.c:160-290       subfield "RAZF", full-flushed 32 KiB blocks, CRC32, ISIZE, big-endian block index
 *   gzip     applet/7gzip.c               one member (the reference: one libdeflate call over the whole file; here the
 *                                         member is a chain of independent 65280-byte pieces, as pigz -i writes them)
 * Host code is plain C over the b200bgzf_* C ABI; b200bgzf_container_frame() needs no GPU (the CPU tests drive it with
 * pieces from the thread emulator and hand the result to the reference's decoders).
 */
#include <stdlib.h>
#include <string.h>
#include <stdio.h>

#include "../../include/b200bgzf.h"
#include "../csrc/bgzf_gzip_route.h"

#define PIECE_MAX 65280u          /* the BGZF rule (applet/7bgzf.c:146-147): a stored piece and its framing fit 64 KiB */
#define DICTZIP_MAX_CHUNKS 32762u /* (0xffff - 10) / 2: the chunk table must fit XLEN (applet/7dictzip.c:178) */
#define ONE_MEMBER 0xffffffffu

/* ---- CRC-32 of a concatenation (polynomial arithmetic on reflected 32-bit words: bit 31 is x^0) ---- */
static uint32_t mulmodp(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (int i = 0; i < 32; i++) {
        if (a & (0x80000000u >> i)) p ^= b;
        b = (b >> 1) ^ ((b & 1u) ? 0xEDB88320u : 0u);          /* b *= x */
    }
    return p;
}

/* x^(8 n) mod P */
static uint32_t xpow8(uint64_t n)
{
    uint32_t r = 0x80000000u, sq = 0x00800000u;                 /* 1, x^8 */
    for (; n; n >>= 1) {
        if (n & 1u) r = mulmodp(r, sq);
        sq = mulmodp(sq, sq);
    }
    return r;
}

uint32_t b200bgzf_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b)
{
    /* CRC(A||B) = CRC(A) * x^(8 len B) + CRC(B)  (mod P), the conditioning of both ends cancels */
    return mulmodp(xpow8(len_b), crc_a) ^ crc_b;
}

static void put16(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
static void put32(uint8_t *p, uint32_t v) { put16(p, v); put16(p + 2, v >> 16); }
static void put32be(uint8_t *p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; }
static void put64be(uint8_t *p, uint64_t v) { put32be(p, (uint32_t)(v >> 32)); put32be(p + 4, (uint32_t)v); }

static uint32_t migz_member_bytes(uint32_t kib) { return (kib ? kib : 512u) * 1024u; }

int b200bgzf_container_plan(int kind, uint32_t param, uint32_t *block_size, b200bgzf_piece_spec *spec)
{
    if (!block_size || !spec) return B200BGZF_E_ARG;
    memset(spec, 0, sizeof *spec);
    switch (kind) {
    case B200BGZF_CONTAINER_GZIP:
        /* one member.  Default: 48 KiB pieces whose matches reach into the 16 KiB before them (dictionary priming, what pigz
         * does between its chunks: -1.6 ... -3 % size against independent 64 KiB pieces for three quarters of the
         * throughput; 32 KiB + 32 KiB compresses no better on FASTQ / SAM text — larger pieces make up for the shorter reach —
         * and is a third slower); B200BGZF_PARAM_INDEPENDENT: independent 65280-byte pieces (pigz -i) */
        spec->member_blocks = ONE_MEMBER; spec->head_gap = 10; spec->tail_gap = 8;
        if (param & B200BGZF_PARAM_INDEPENDENT) {
            *block_size = PIECE_MAX;
        } else {
            *block_size = 49152u;
            spec->history = 16320u;
        }
        return B200BGZF_OK;
    case B200BGZF_CONTAINER_MIGZ: {
        const uint32_t kib = param & ~(B200BGZF_PARAM_SAFE | B200BGZF_PARAM_PRIMED);
        if (kib > 4u * 1024u * 1024u - 1u) return B200BGZF_E_ARG;             /* ISIZE and the MZ field are 32 bits */
        const uint32_t m = migz_member_bytes(kib);
        /* the fewest equal pieces that make up a member exactly: of at most 65536 bytes (512 KiB = 8 x 64 KiB; a piece that
         * does not compress at all then overflows its slot and the call reports B200BGZF_E_NOFIT), or, with
         * B200BGZF_PARAM_SAFE, of at most 65280 bytes so that even a stored piece fits (512 KiB = 16 x 32 KiB) */
        /* B200BGZF_PARAM_PRIMED: pieces of at most 32 KiB whose matches reach into the 32 KiB before them inside the member */
        const uint32_t most = (param & B200BGZF_PARAM_PRIMED) ? 65536u - B200BGZF_MAX_HISTORY : (param & B200BGZF_PARAM_SAFE) ? PIECE_MAX : 65536u;
        uint32_t k = (m + most - 1u) / most;
        while (m % k) k++;
        if ((param & B200BGZF_PARAM_PRIMED) && k > 1) spec->history = B200BGZF_MAX_HISTORY;
        *block_size = m / k;
        spec->member_blocks = k; spec->head_gap = 20; spec->tail_gap = 8;
        return B200BGZF_OK;
    }
    case B200BGZF_CONTAINER_GZINGA:
        *block_size = 51200u;                                                   /* 100 KiB members (7gzinga.c:79) */
        spec->member_blocks = 2; spec->head_gap = 11; spec->tail_gap = 8;
        return B200BGZF_OK;
    case B200BGZF_CONTAINER_DICTZIP:
        if (param > PIECE_MAX) return B200BGZF_E_ARG;
        *block_size = param ? param : 58315u;                                   /* 7dictzip.c:550-551 */
        spec->member_blocks = ONE_MEMBER; spec->tail_gap = 10; spec->no_final = 1;
        return B200BGZF_OK;
    case B200BGZF_CONTAINER_RAZF:
        *block_size = 32768u;                                                   /* 7razf.c:165 */
        spec->member_blocks = ONE_MEMBER; spec->head_gap = 19; spec->tail_gap = 8;
        return B200BGZF_OK;
    }
    return B200BGZF_E_ARG;
}

size_t b200bgzf_container_head(int kind, size_t npieces) { return kind == B200BGZF_CONTAINER_DICTZIP ? 22u + 2u * npieces : 0u; }

size_t b200bgzf_container_bound(int kind, uint32_t param, size_t in_bytes)
{
    uint32_t bs;
    b200bgzf_piece_spec sp;
    if (b200bgzf_container_plan(kind, kind == B200BGZF_CONTAINER_MIGZ ? param | B200BGZF_PARAM_SAFE : param, &bs, &sp) != 0) return 0;
    const size_t np = (in_bytes + bs - 1) / bs;                                 /* (the plan with the most pieces) */
    size_t extra = 64;
    if (kind == B200BGZF_CONTAINER_GZINGA) extra += 32 + 34 * ((np + 1) / 2);   /* "n:offset;" per member */
    if (kind == B200BGZF_CONTAINER_RAZF) extra += 4 * np + 64;
    if (kind == B200BGZF_CONTAINER_DICTZIP) extra += 2 * np + 64 * (np / DICTZIP_MAX_CHUNKS + 1);
    return b200bgzf_compress_bound(in_bytes, bs) + b200bgzf_pieces_gap_bytes(in_bytes, bs, &sp) + extra;
}

/* CRC-32 and byte count of the input behind pieces [f, l]; shift = x^(8 bs): all pieces but the stream's last are bs bytes long */
static uint32_t span_crc(const uint32_t *crc, size_t f, size_t l, size_t npieces, uint32_t bs, uint32_t shift, size_t in_bytes, uint64_t *bytes)
{
    uint32_t c = 0;
    uint64_t n = 0;
    for (size_t i = f; i <= l; i++) {
        const uint64_t len = i + 1 == npieces ? in_bytes - (uint64_t)i * bs : bs;
        c = i == f ? crc[i] : len == bs ? mulmodp(shift, c) ^ crc[i] : b200bgzf_crc32_combine(c, crc[i], len);
        n += len;
    }
    *bytes = n;
    return c;
}

size_t b200bgzf_container_frame(int kind, uint32_t param, void *member, size_t cap, size_t stream_bytes, const uint64_t *piece_off,
                                const uint32_t *piece_crc, size_t npieces, size_t in_bytes)
{
    uint32_t bs;
    b200bgzf_piece_spec sp;
    uint8_t *o = (uint8_t *)member;
    if (!o || b200bgzf_container_plan(kind, param, &bs, &sp) != 0) return 0;
    if (npieces && (!piece_off || !piece_crc)) return 0;
    if (npieces != (in_bytes + bs - 1) / bs) return 0;
    uint64_t nbytes = 0;
    const uint32_t shift = xpow8(bs);

    if (kind == B200BGZF_CONTAINER_DICTZIP) {
        if (npieces > DICTZIP_MAX_CHUNKS) return 0;
        const size_t head = b200bgzf_container_head(kind, npieces);
        size_t end = head + stream_bytes;
        if (npieces == 0) end = head + 10;                       /* an empty member still closes its DEFLATE stream */
        if (cap < end) return 0;
        static const uint8_t h10[10] = { 0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0x03 };
        memcpy(o, h10, 10);
        put16(o + 10, (uint32_t)(10 + 2 * npieces));
        o[12] = 'R'; o[13] = 'A';
        put16(o + 14, (uint32_t)(6 + 2 * npieces));
        put16(o + 16, 1);
        put16(o + 18, bs);
        put16(o + 20, (uint32_t)npieces);
        for (size_t i = 0; i < npieces; i++) {
            const uint64_t next = i + 1 < npieces ? piece_off[i + 1] : stream_bytes - 10;
            const uint64_t sz = next - piece_off[i];
            if (sz > 0xffffu) return 0;
            put16(o + 22 + 2 * i, (uint32_t)sz);
        }
        const uint32_t crc = npieces ? span_crc(piece_crc, 0, npieces - 1, npieces, bs, shift, in_bytes, &nbytes) : 0u;
        o[end - 10] = 0x03; o[end - 9] = 0x00;                   /* "null deflation to conform normal gzip" (7dictzip.c:311) */
        put32(o + end - 8, crc);
        put32(o + end - 4, (uint32_t)in_bytes);
        return end;
    }

    if (npieces == 0) {
        /* empty input: only the whole-file containers write anything */
        if (kind == B200BGZF_CONTAINER_MIGZ) return 0;
        if (kind == B200BGZF_CONTAINER_GZIP || kind == B200BGZF_CONTAINER_RAZF) {
            const size_t need = sp.head_gap + 2u + 8u;
            if (cap < need + 64) return 0;
            memset(o, 0, need);
            o[sp.head_gap] = 0x03;
            stream_bytes = need;
        }
    }
    if (cap < stream_bytes) return 0;
    size_t pos = stream_bytes;

    /* the members: header into the head gap, CRC32 + ISIZE into the tail gap */
    const size_t k = sp.member_blocks;
    for (size_t f = 0; f < npieces; f += k) {
        const size_t l = (npieces - f > k ? f + k : npieces) - 1;
        const uint64_t start = piece_off[f], end = l + 1 < npieces ? piece_off[l + 1] : stream_bytes;
        if (end < start + sp.head_gap + sp.tail_gap || end > stream_bytes) return 0;
        uint8_t *h = o + start;
        const uint32_t crc = span_crc(piece_crc, f, l, npieces, bs, shift, in_bytes, &nbytes);
        switch (kind) {
        case B200BGZF_CONTAINER_MIGZ: {
            static const uint8_t hd[16] = { 0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x08, 0, 'M', 'Z', 0x04, 0 };
            memcpy(h, hd, 16);
            put32(h + 16, (uint32_t)(end - start - 28));
            break;
        }
        case B200BGZF_CONTAINER_GZINGA: {
            static const uint8_t hd[11] = { 0x1f, 0x8b, 0x08, 0x10, 0, 0, 0, 0, 0, 0xff, 0 };
            memcpy(h, hd, 11);
            break;
        }
        case B200BGZF_CONTAINER_RAZF: {
            static const uint8_t hd[19] = { 0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0x03, 0x07, 0, 'R', 'A', 'Z', 'F', 0x01, 0x80, 0x00 };
            memcpy(h, hd, 19);
            break;
        }
        default: {
            static const uint8_t hd[10] = { 0x1f, 0x8b, 0x08, 0x00, 0, 0, 0, 0, 0, 0xff };
            memcpy(h, hd, 10);
            break;
        }
        }
        put32(o + end - 8, crc);
        put32(o + end - 4, (uint32_t)nbytes);
    }
    if (npieces == 0 && kind == B200BGZF_CONTAINER_GZIP) {
        static const uint8_t hd[10] = { 0x1f, 0x8b, 0x08, 0x00, 0, 0, 0, 0, 0, 0xff };
        memcpy(o, hd, 10);
    }
    if (npieces == 0 && kind == B200BGZF_CONTAINER_RAZF) {
        static const uint8_t hd[19] = { 0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0x03, 0x07, 0, 'R', 'A', 'Z', 'F', 0x01, 0x80, 0x00 };
        memcpy(o, hd, 19);
    }

    if (kind == B200BGZF_CONTAINER_GZINGA) {
        /* the index member: header, comment "0:end0;1:end1;...", NUL, an empty static block, CRC32 0, ISIZE 0 (7gzinga.c:207-211) */
        static const uint8_t hd[10] = { 0x1f, 0x8b, 0x08, 0x10, 0, 0, 0, 0, 0, 0xff };
        const size_t members = (npieces + k - 1) / k;
        if (cap < pos + 10 + 34 * members + 11) return 0;
        memcpy(o + pos, hd, 10);
        pos += 10;
        for (size_t m = 0; m < members; m++) {
            const size_t nf = (m + 1) * k;
            const uint64_t end = nf < npieces ? piece_off[nf] : stream_bytes;
            pos += (size_t)sprintf((char *)o + pos, "%llu:%llu;", (unsigned long long)m, (unsigned long long)end);
        }
        static const uint8_t tl[11] = { 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
        memcpy(o + pos, tl, 11);
        pos += 11;
    }
    if (kind == B200BGZF_CONTAINER_RAZF) {
        /* the block index (7razf.c:166-171,262-275): u32 count of the blocks after the first, u64 start of bin 0 (= of the
         * second block), u32 start of every later block relative to it, then the input size and where the index begins */
        if (in_bytes >> 32) return 0;
        const size_t tb = npieces ? npieces - 1 : 0;
        if (cap < pos + 4 + 8 + 4 * tb + 16) return 0;
        const uint64_t index_at = pos, bin0 = tb ? piece_off[1] : 0;
        put32be(o + pos, (uint32_t)tb);
        put64be(o + pos + 4, bin0);
        pos += 12;
        for (size_t i = 0; i < tb; i++, pos += 4) put32be(o + pos, (uint32_t)(piece_off[i + 1] - bin0));
        put64be(o + pos, in_bytes);
        put64be(o + pos + 8, index_at);
        pos += 16;
    }
    return pos;
}

int b200bgzf_container_compress_host(b200bgzf_ctx *ctx, int kind, uint32_t param, const void *in, size_t in_bytes, int level,
                                     void *out, size_t out_cap, size_t *out_bytes)
{
    uint32_t bs;
    b200bgzf_piece_spec sp;
    if (!ctx || !out || !out_bytes || (!in && in_bytes)) return B200BGZF_E_ARG;
    if (b200bgzf_container_plan(kind, param, &bs, &sp) != 0) return B200BGZF_E_ARG;
    if (kind == B200BGZF_CONTAINER_RAZF && (in_bytes >> 32)) return B200BGZF_E_ARG;
    if (out_cap < b200bgzf_container_bound(kind, param, in_bytes)) return B200BGZF_E_NOSPACE;
    *out_bytes = 0;
    /* dictzip: one call per member of at most 32762 chunks; the others: one call */
    const size_t np_total = (in_bytes + bs - 1) / bs;
    const size_t per_call = kind == B200BGZF_CONTAINER_DICTZIP ? DICTZIP_MAX_CHUNKS : (np_total ? np_total : 1);
    uint64_t *off = (uint64_t *)malloc(sizeof(uint64_t) * (per_call < np_total ? per_call : np_total) + 8);
    uint32_t *crc = (uint32_t *)malloc(sizeof(uint32_t) * (per_call < np_total ? per_call : np_total) + 8);
    if (!off || !crc) { free(off); free(crc); return B200BGZF_E_ARG; }
    int rc = B200BGZF_OK;
    size_t pos = 0, done = 0;
    do {
        const size_t np = np_total - done < per_call ? np_total - done : per_call;
        const size_t byte0 = done * bs, bytes = (done + np) * bs < in_bytes ? np * (size_t)bs : in_bytes - byte0;
        const size_t head = b200bgzf_container_head(kind, np);
        size_t stream = 0;
        if (np) {
            rc = b200bgzf_compress_pieces_host(ctx, (const uint8_t *)in + byte0, bytes, bs, level, &sp, (uint8_t *)out + pos + head,
                                               out_cap - pos - head, &stream, off, crc, np);
            if (rc != 0) break;
        }
        const size_t total = b200bgzf_container_frame(kind, param, (uint8_t *)out + pos, out_cap - pos, stream, off, crc, np, bytes);
        if (!total && !(kind == B200BGZF_CONTAINER_MIGZ && np == 0)) { rc = B200BGZF_E_NOSPACE; break; }
        pos += total;
        done += np;
    } while (done < np_total);
    free(off);
    free(crc);
    if (rc == B200BGZF_E_NOFIT && kind == B200BGZF_CONTAINER_MIGZ && !(param & B200BGZF_PARAM_SAFE))
        /* a 64 KiB piece that does not compress overflows its slot: redo the file with pieces that always fit (the reference's
         * BGZF writer does the same with its 0x10000-byte blocks, applet/7bgzf.c:256-262) */
        return b200bgzf_container_compress_host(ctx, kind, param | B200BGZF_PARAM_SAFE, in, in_bytes, level, out, out_cap, out_bytes);
    if (rc == 0) *out_bytes = pos;
    return rc;
}

/* ================================================================================================================
 * Readers: the unit lists of the indexed containers (no GPU involved), then one b200bgzf_inflate_units_host() call.
 * ================================================================================================================ */
static uint32_t get16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
static uint32_t get32(const uint8_t *p) { return get16(p) | (get16(p + 2) << 16); }
static uint64_t get32be(const uint8_t *p) { return ((uint64_t)p[0] << 24) | ((uint64_t)p[1] << 16) | ((uint64_t)p[2] << 8) | p[3]; }
static uint64_t get64be(const uint8_t *p) { return (get32be(p) << 32) | get32be(p + 4); }

/* RFC 1952 header: returns its length (0: not a gzip member / cut short) and where the extra field lies */
static size_t gz_header(const uint8_t *p, size_t avail, size_t *xoff, size_t *xlen)
{
    if (avail < 10 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || (p[3] & 0xE0u)) return 0;
    size_t n = 10;
    *xoff = 0;
    *xlen = 0;
    if (p[3] & 0x04u) {
        if (avail < n + 2) return 0;
        *xlen = get16(p + n);
        n += 2;
        *xoff = n;
        if (avail < n + *xlen) return 0;
        n += *xlen;
    }
    for (int f = 0x08; f <= 0x10; f <<= 1)
        if (p[3] & f) {
            while (n < avail && p[n]) n++;
            if (n >= avail) return 0;
            n++;
        }
    if (p[3] & 0x02u) n += 2;
    return n <= avail ? n : 0;
}

size_t bgzf_gz_header(const uint8_t *p, size_t avail, size_t *xoff, size_t *xlen) { return gz_header(p, avail, xoff, xlen); }

/* a member made of pieces: units [first, first + count) together must have the CRC-32 its trailer states */
struct member_check {
    size_t first, count;
    uint32_t crc;
};
struct unit_list {
    b200bgzf_unit *u;
    size_t n, cap;
    uint64_t out_bytes;
    struct member_check *chk;
    size_t nchk, chk_cap;
};
static int check_push(struct unit_list *l, size_t first, size_t count, uint32_t crc)
{
    if (l->nchk == l->chk_cap) {
        const size_t cap = l->chk_cap ? l->chk_cap * 2 : 16;
        struct member_check *c = (struct member_check *)realloc(l->chk, cap * sizeof *c);
        if (!c) return -1;
        l->chk = c;
        l->chk_cap = cap;
    }
    l->chk[l->nchk].first = first;
    l->chk[l->nchk].count = count;
    l->chk[l->nchk].crc = crc;
    l->nchk++;
    return 0;
}
static int unit_push(struct unit_list *l, uint64_t in_off, uint64_t in_len, uint32_t hdr_len, uint64_t out_len, int piece)
{
    if (in_len == 0 || in_len > 0xffffffffull || out_len > 0xffffffffull) return -1;
    if (l->n == l->cap) {
        const size_t cap = l->cap ? l->cap * 2 : 1024;
        b200bgzf_unit *u = (b200bgzf_unit *)realloc(l->u, cap * sizeof *u);
        if (!u) return -1;
        l->u = u;
        l->cap = cap;
    }
    b200bgzf_unit *x = &l->u[l->n++];
    x->in_off = in_off;
    x->in_len = (uint32_t)in_len;
    x->hdr_len = hdr_len;
    x->out_len = (uint32_t)out_len;
    x->piece = piece ? 1u : 0u;
    l->out_bytes += out_len;
    return 0;
}

/* dictzip (applet/7dictzip.c:136-175,320-400): members follow one another; each lists its chunks in the "RA" subfield */
static int units_dictzip(const uint8_t *p, size_t n, struct unit_list *l)
{
    size_t pos = 0;
    while (pos < n) {
        size_t xoff, xlen;
        const size_t h = gz_header(p + pos, n - pos, &xoff, &xlen);
        if (!h || xlen < 10) return B200BGZF_E_FORMAT;
        const uint8_t *x = p + pos + xoff;
        if (x[0] != 'R' || x[1] != 'A' || get16(x + 2) + 4 != xlen || get16(x + 4) != 1) return B200BGZF_E_FORMAT;
        const uint32_t chlen = get16(x + 6), chcnt = get16(x + 8);
        if (chcnt * 2u + 10u != xlen || (chcnt && !chlen)) return B200BGZF_E_FORMAT;
        uint64_t data = 0;
        for (uint32_t i = 0; i < chcnt; i++) data += get16(x + 10 + 2 * i);
        /* after the chunks: the closing empty block (03 00; some writers end the last chunk with the final block and have no
         * such bytes), CRC32, ISIZE */
        size_t at = pos + h + data;
        if (at + 8 > n) return B200BGZF_E_FORMAT;
        if (at + 10 <= n && p[at] == 0x03 && p[at + 1] == 0x00) at += 2;
        const uint64_t isize = get32(p + at + 4);
        if (chcnt && (isize > (uint64_t)chcnt * chlen || isize + chlen <= (uint64_t)chcnt * chlen)) return B200BGZF_E_FORMAT;
        uint64_t off = pos + h;
        if (chcnt && check_push(l, l->n, chcnt, get32(p + at))) return B200BGZF_E_FORMAT;
        for (uint32_t i = 0; i < chcnt; i++) {
            const uint32_t sz = get16(x + 10 + 2 * i);
            const uint64_t outl = i + 1 < chcnt ? chlen : isize - (uint64_t)(chcnt - 1) * chlen;
            if (unit_push(l, off, sz, 0, outl, 1)) return B200BGZF_E_FORMAT;
            off += sz;
        }
        pos = at + 8;
    }
    return B200BGZF_OK;
}

/* RAZF (applet/7razf.c:293-384): block size in the header's subfield, block index (big endian) located by the last 16 bytes */
static int units_razf(const uint8_t *p, size_t n, struct unit_list *l)
{
    size_t xoff, xlen;
    const size_t h = gz_header(p, n, &xoff, &xlen);
    if (!h || xlen < 7 || memcmp(p + xoff, "RAZF", 4) || n < h + 8 + 12 + 16) return B200BGZF_E_FORMAT;
    const uint32_t bs = ((uint32_t)p[xoff + 5] << 8) | p[xoff + 6];
    const uint64_t fsize = get64be(p + n - 16), index_at = get64be(p + n - 8);
    if (!bs || index_at < h + 8 || index_at + 12 + 16 > n) return B200BGZF_E_FORMAT;
    const uint64_t tb = get32be(p + index_at);
    const uint64_t binsize = (1ull << 32) / bs, bins = tb / binsize;
    const uint64_t cells_at = index_at + 4 + 8 * (bins + 1);
    if (cells_at + 4 * tb + 16 != n) return B200BGZF_E_FORMAT;
    if (fsize == 0) return B200BGZF_OK;
    if (tb + 1 != (fsize + bs - 1) / bs) return B200BGZF_E_FORMAT;
    uint64_t start = h;
    if (check_push(l, 0, (size_t)tb + 1, get32(p + index_at - 8))) return B200BGZF_E_FORMAT;
    for (uint64_t i = 0; i <= tb; i++) {
        uint64_t next = index_at - 8;                                        /* the last block ends at the trailer */
        if (i < tb) next = get64be(p + index_at + 4 + 8 * (i / binsize)) + get32be(p + cells_at + 4 * i);
        if (next <= start || next > index_at - 8) return B200BGZF_E_FORMAT;
        const uint64_t outl = i < tb ? bs : fsize - tb * bs;
        if (unit_push(l, start, next - start, 0, outl, 1)) return B200BGZF_E_FORMAT;
        start = next;
    }
    return B200BGZF_OK;
}

/* GZinga (applet/7gzinga.c:218-260): the last member's comment lists where every data member ends */
static int units_gzinga(const uint8_t *p, size_t n, struct unit_list *l)
{
    static const uint8_t sig[10] = { 0x1f, 0x8b, 0x08, 0x10, 0, 0, 0, 0, 0, 0xff };
    static const uint8_t tail[11] = { 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
    if (n < 21 || memcmp(p + n - 11, tail, 11)) return B200BGZF_E_FORMAT;
    /* the index member: the last header whose comment is "digits:digits;" all the way to that tail */
    size_t idx = n;
    for (size_t at = n - 21;; at--) {
        if (!memcmp(p + at, sig, 10)) {
            size_t k = at + 10;
            while (k < n - 11 && ((p[k] >= '0' && p[k] <= '9') || p[k] == ':' || p[k] == ';')) k++;
            if (k == n - 11) { idx = at; break; }
        }
        if (at == 0) break;
    }
    if (idx == n) return B200BGZF_E_FORMAT;
    uint64_t start = 0;
    for (size_t k = idx + 10; k < n - 11;) {
        while (k < n - 11 && p[k] != ':') k++;                               /* member number */
        uint64_t end = 0;
        for (k++; k < n - 11 && p[k] != ';'; k++) end = end * 10 + (uint64_t)(p[k] - '0');
        k++;
        if (end <= start || end > idx) return B200BGZF_E_FORMAT;
        size_t xoff, xlen;
        const size_t h = gz_header(p + start, end - start, &xoff, &xlen);
        if (!h || end - start < h + 8) return B200BGZF_E_FORMAT;
        if (unit_push(l, start, end - start, (uint32_t)h, get32(p + end - 4), 0)) return B200BGZF_E_FORMAT;
        start = end;
    }
    return start == idx ? B200BGZF_OK : B200BGZF_E_FORMAT;
}

/* plain gzip: one unit spanning the input (b200bgzf_container_inflate_host decodes it between its flush points where it has
 * them, else on one warp) */
static int units_gzip(const uint8_t *p, size_t n, struct unit_list *l)
{
    /* without an index a member's end is only known once it is decoded: a single member is taken to span the input */
    size_t xoff, xlen;
    const size_t h = gz_header(p, n, &xoff, &xlen);
    if (!h || n < h + 8 + 2) return B200BGZF_E_FORMAT;
    return unit_push(l, 0, n, (uint32_t)h, get32(p + n - 4), 0) ? B200BGZF_E_FORMAT : B200BGZF_OK;
}

static int list_units(int kind, const void *in, size_t in_bytes, struct unit_list *l)
{
    memset(l, 0, sizeof *l);
    switch (kind) {
    case B200BGZF_CONTAINER_DICTZIP: return units_dictzip((const uint8_t *)in, in_bytes, l);
    case B200BGZF_CONTAINER_RAZF: return units_razf((const uint8_t *)in, in_bytes, l);
    case B200BGZF_CONTAINER_GZINGA: return units_gzinga((const uint8_t *)in, in_bytes, l);
    case B200BGZF_CONTAINER_GZIP: return units_gzip((const uint8_t *)in, in_bytes, l);
    }
    return B200BGZF_E_ARG;
}

int b200bgzf_container_units(int kind, const void *in, size_t in_bytes, b200bgzf_unit **units, size_t *nunits, size_t *out_bytes)
{
    if (!in || !units || !nunits) return B200BGZF_E_ARG;
    if (in_bytes == 0) return B200BGZF_E_FORMAT;
    struct unit_list l;
    const int rc = list_units(kind, in, in_bytes, &l);
    free(l.chk);
    if (rc != 0) {
        free(l.u);
        return rc;
    }
    *units = l.u;
    *nunits = l.n;
    if (out_bytes) *out_bytes = (size_t)l.out_bytes;
    return B200BGZF_OK;
}

void b200bgzf_units_free(b200bgzf_unit *units) { free(units); }

/* members that carry their own size (BGZF, MiGz, mgzip) are found by the header walk and decoded one warp each; `7gzip -d`
 * takes that route too when its input turns out to be such a stream */
static int sized_members(int kind, const void *in, size_t in_bytes, size_t *out_bytes, size_t *nmembers)
{
    if (kind != B200BGZF_CONTAINER_MIGZ && kind != B200BGZF_CONTAINER_GZIP) return 0;
    return b200bgzf_inflate_size_host(in, in_bytes, out_bytes, nmembers) == 0;
}

int b200bgzf_container_inflate_size(int kind, const void *in, size_t in_bytes, size_t *out_bytes, size_t *nunits)
{
    size_t total = 0, n = 0;
    if (!in || !out_bytes) return B200BGZF_E_ARG;
    if (!sized_members(kind, in, in_bytes, &total, &n)) {
        if (kind == B200BGZF_CONTAINER_MIGZ) return B200BGZF_E_FORMAT;
        b200bgzf_unit *u = NULL;
        const int rc = b200bgzf_container_units(kind, in, in_bytes, &u, &n, &total);
        if (rc != 0) return rc;
        free(u);
    }
    *out_bytes = total;
    if (nunits) *nunits = n;
    return B200BGZF_OK;
}

int b200bgzf_container_inflate_host(b200bgzf_ctx *ctx, int kind, const void *in, size_t in_bytes, void *out, size_t out_cap, size_t *out_bytes,
                                    unsigned flags)
{
    size_t sized_total = 0, sized_n = 0;
    if (kind == B200BGZF_CONTAINER_MIGZ || (in && sized_members(kind, in, in_bytes, &sized_total, &sized_n)))
        return b200bgzf_inflate_host(ctx, in, in_bytes, out, out_cap, out_bytes, flags);
    if (!in || in_bytes == 0) return in ? B200BGZF_E_FORMAT : B200BGZF_E_ARG;
    struct unit_list l;
    int rc = list_units(kind, in, in_bytes, &l);
    uint32_t *crc = NULL;
    if (rc == 0) {
        if (out_bytes) *out_bytes = (size_t)l.out_bytes;
        /* B200BGZF_VERIFY: members are checked against their trailers on the device; the CRC-32 of a member made of pieces
         * (dictzip, RAZF) is combined here from those of its pieces (the reference's readers check neither) */
        if ((flags & B200BGZF_VERIFY) && l.nchk && !(crc = (uint32_t *)malloc(sizeof(uint32_t) * (l.n + 1)))) rc = B200BGZF_E_ARG;
        else if (l.out_bytes > out_cap) rc = B200BGZF_E_NOSPACE;
        else {
            /* whole-stream gzip: in parallel between the member's flush points when it has a complete chain of them */
            rc = kind == B200BGZF_CONTAINER_GZIP && l.n == 1
                     ? bgzf_gzip_inflate_host(ctx, in, in_bytes, l.u[0].hdr_len, out, out_cap, out_bytes, flags)
                     : BGZF_GZIP_FALLBACK;
            if (rc == BGZF_GZIP_FALLBACK) rc = b200bgzf_inflate_units_host(ctx, in, in_bytes, l.u, l.n, out, out_cap, out_bytes, flags, crc);
        }
    }
    if (rc == 0 && crc)
        for (size_t k = 0; k < l.nchk && rc == 0; k++) {
            uint32_t c = 0;
            for (size_t i = 0; i < l.chk[k].count; i++) {
                const size_t ui = l.chk[k].first + i;
                c = i ? b200bgzf_crc32_combine(c, crc[ui], l.u[ui].out_len) : crc[ui];
            }
            if (c != l.chk[k].crc) rc = B200BGZF_E_CRC;
        }
    free(crc);
    free(l.u);
    free(l.chk);
    return rc;
}
