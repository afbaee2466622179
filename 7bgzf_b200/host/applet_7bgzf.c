/*
 * applet_7bgzf.c — the `7bgzf` command line of the reference (applet/7bgzf.c:371-551), driving the GPU codec.
 *
 *   7bgzf -c -l6 [-@ N] < in > out.bgz        compress (stdin -> stdout only)
 *   7bgzf -d [-@ N] < in.bgz > out            decompress
 *   7bgzf -d --offset=N [--size=M] [--gzi=F] < in.bgz > out    decompress bytes [N, N+M) only (bgzip -b N -s M)
 *   7bgzf --reindex --gzi=F < in.bgz          write the .gzi of an existing stream (bgzip -r)
 *   7gzip --reindex --index=F < in.gz         write the checkpoint index of a whole-stream gzip member
 *   7gzip -d --offset=N [--size=M] --index=F < in.gz > out    decompress bytes [N, N+M) only, through that index
 *
 * Same flags as the reference's popt table (7bgzf.c:379-398): -l[N]/--libdeflate[=N] (1-12, default 6),
 * -z -m -s -S -n -C -i -K -T [N] and -Z N (the other method flags: each selects a level for the one GPU codec,
 * there is no multi-backend dispatch), -@ N/--threads (accepted; the GPU path is always block-parallel),
 * -d/--decompress, -c/--stdout (ignored).  Exactly one method unless -d (7bgzf.c:467-479); refuses a
 * terminal on stdin or stdout (:491,498); stderr carries the reference's lines:
 *   "compression level = %d (libdeflate)", "%d done.", "ellapsed time: %.6f sec".
 * Payload blocks are always 0xff00 bytes (the reference's multi-thread rule, 7bgzf.c:141-147).
 *
 * Where the reference creates a thread per block, this applet runs a three-stage pipeline over page-locked
 * slots: a reader thread (stdin -> slot), the calling thread (slot -> GPU codec -> slot), a writer thread
 * (slot -> stdout), so file I/O, PCIe copies and kernels overlap.
 * Host code is C; CUDA is reached only through the b200bgzf_* C ABI.  No GPU => error, no CPU fallback.
 */
#include <getopt.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>

#include "../../include/b200bgzf.h"

#define SLOT_BLOCKS 1024u                     /* 63.75 MiB of payload per slot */
#define NSLOTS 3

struct method_flag {
    char short_opt;
    const char *label;
    int default_level;
};

static const struct method_flag k_flags[] = {
    { 'z', "zlib", 6 },   { 'm', "miniz", 1 },    { 's', "slz", 1 },     { 'l', "libdeflate", 6 }, { 'S', "7zip", 2 },  { 'n', "zlibng", 6 },
    { 'C', "cryptopp", 6 }, { 'i', "igzip", 1 },  { 'K', "kzip", 1 },    { 'Z', "zopfli", 0 },     { 'T', "store", 1 },
};
#define NFLAGS (sizeof k_flags / sizeof k_flags[0])

static void usage(const char *argv0)
{
    fprintf(stderr,
            "Usage: %s -cz9 < dec.bin > enc.bgz or -cd < enc.bgz > dec.bin\n"
            "  -c, --stdout              stdout (currently ignored; always output to stdout)\n"
            "  -z, --zlib[=level]        1-9 (default 6) zlib\n"
            "  -m, --miniz[=level]       1-9 (default 1) miniz\n"
            "  -s, --slz[=level]         1-1 (default 1) slz\n"
            "  -l, --libdeflate[=level]  1-12 (default 6) libdeflate\n"
            "  -S, --7zip[=level]        1-9 (default 2) 7zip\n"
            "  -n, --zlibng[=level]      1-9 (default 6) zlibng\n"
            "  -C, --cryptopp[=level]    1-9 (default 6) cryptopp\n"
            "  -i, --igzip[=level]       1-4 (default 1) igzip\n"
            "  -K, --kzip[=level]        1-1 (default 1) kzip\n"
            "  -Z, --zopfli=numiterations zopfli\n"
            "  -T, --store[=level]       1-1 (default 1) store\n"
            "  -@, --threads=threads     threads\n"
            "  -d, --decompress          decompress\n"
            "      --gzi=FILE            (extension) also write a bgzip-style .gzi index of the members to FILE\n"
            "      --offset=N            (extension, with -d) decompress from byte N of the data on (read --gzi=FILE if given)\n"
            "      --size=M              (extension, with --offset) at most M bytes\n"
            "      --reindex             (extension) write the .gzi of the stream on stdin to --gzi=FILE, nothing to stdout\n"
            "      --index=FILE          (extension, 7gzip) the checkpoint index: written by --reindex, read by -d --offset (required)\n"
            "      --devices=N           (extension) spread the blocks over N GPUs (contiguous block ranges, same output)\n"
            "      --independent         (extension, 7gzip) pieces without the 16 KiB of history before them: faster, 2-3 %% larger\n"
            "      --primed              (extension, 7migz) pieces of a member see the 32 KiB before them: slower, 2 %% smaller\n"
            "\nNote: every method runs on the B200 BGZF codec (libdeflate level classes 1-12).\n",
            argv0);
}

/* ---- a tiny ordered three-stage pipeline ---- */
enum { EMPTY = 0, FILLED, DONE };
struct slot {
    unsigned char *in, *out;
    size_t in_len, out_len, members;
    int state, last;
};
struct pipe_state {
    struct slot s[NSLOTS];
    pthread_mutex_t mu;
    pthread_cond_t cv;
    FILE *fin, *fout;
    size_t in_cap, out_cap;
    int decompress, failed;
};

static void set_state(struct pipe_state *ps, struct slot *sl, int st)
{
    pthread_mutex_lock(&ps->mu);
    sl->state = st;
    pthread_cond_broadcast(&ps->cv);
    pthread_mutex_unlock(&ps->mu);
}
static void wait_state(struct pipe_state *ps, struct slot *sl, int st)
{
    pthread_mutex_lock(&ps->mu);
    while (sl->state != st && !ps->failed) pthread_cond_wait(&ps->cv, &ps->mu);
    pthread_mutex_unlock(&ps->mu);
}
static void fail(struct pipe_state *ps)
{
    pthread_mutex_lock(&ps->mu);
    ps->failed = 1;
    pthread_cond_broadcast(&ps->cv);
    pthread_mutex_unlock(&ps->mu);
}

static double now_s(void)
{
    struct timeval t;
    gettimeofday(&t, NULL);
    return t.tv_sec + t.tv_usec * 1e-6;
}
static double g_t_read, g_t_write, g_t_codec, g_t_alloc, g_t_create;

/* stdin is read with read(2) into the slot; a regular file (`7bgzf -c -l6 < reads.fq`) by four threads at once, each with
 * pread(2) on its quarter of the slot: one thread copies out of the page cache at 2-3 GB/s, which would otherwise be the
 * slowest stage of the pipeline */
#define READ_THREADS 4
static int g_in_regular;
static off_t g_in_pos;
struct pread_job {
    pthread_t th;
    unsigned char *buf;
    size_t want, got;
    off_t off;
};
static void *pread_main(void *arg)
{
    struct pread_job *j = (struct pread_job *)arg;
    j->got = 0;
    while (j->got < j->want) {
        const ssize_t r = pread(0, j->buf + j->got, j->want - j->got, j->off + (off_t)j->got);
        if (r <= 0) break;
        j->got += (size_t)r;
    }
    return NULL;
}
static size_t read_full(FILE *f, unsigned char *buf, size_t want)
{
    (void)f;
    size_t n = 0;
    if (g_in_regular && want >= ((size_t)8 << 20)) {
        struct pread_job jobs[READ_THREADS];
        const size_t part = (want / READ_THREADS + 4095) & ~(size_t)4095;
        for (int i = 0; i < READ_THREADS; i++) {
            const size_t lo = (size_t)i * part < want ? (size_t)i * part : want, hi = lo + part < want ? lo + part : want;
            jobs[i].buf = buf + lo;
            jobs[i].want = hi - lo;
            jobs[i].off = g_in_pos + (off_t)lo;
            if (i == READ_THREADS - 1 || pthread_create(&jobs[i].th, NULL, pread_main, &jobs[i]) != 0) {
                jobs[i].th = 0;
                pread_main(&jobs[i]);
            }
        }
        int short_seen = 0;
        for (int i = 0; i < READ_THREADS; i++) {
            if (jobs[i].th) pthread_join(jobs[i].th, NULL);
            if (!short_seen) n += jobs[i].got;                 /* (bytes after a short part belong to nobody: end of file) */
            if (jobs[i].got < jobs[i].want) short_seen = 1;
        }
        g_in_pos += (off_t)n;
        return n;
    }
    while (n < want) {
        const ssize_t r = g_in_regular ? pread(0, buf + n, want - n, g_in_pos + (off_t)n) : read(0, buf + n, want - n);
        if (r <= 0) break;
        n += (size_t)r;
    }
    g_in_pos += (off_t)n;
    return n;
}

/* whole members at the front of buf[0..have) whose payloads fit in out_cap: bytes used, members, total ISIZE;
 * -1: not a member the reference's loop would accept (7bgzf.c:81-131: BGZF, MiGz, mgzip), -2: one member alone is
 * larger than a slot */
static long whole_members(const unsigned char *buf, size_t have, size_t in_cap, size_t out_cap, int at_eof, size_t *nm, size_t *isize_total)
{
    size_t used = 0;
    *nm = 0;
    *isize_total = 0;
    while (used < have) {
        const unsigned char *p = buf + used;
        uint64_t sz = 0;
        if (!b200bgzf_member_header(p, have - used, &sz)) {
            /* either garbage, or a member that continues beyond what has been read so far */
            if (have - used >= 2 && (p[0] != 0x1f || p[1] != 0x8b)) return -1;
            if (!at_eof && have - used < in_cap && *nm > 0) break;
            if (!at_eof && *nm == 0 && have - used >= in_cap) return -2;
            if (at_eof || *nm == 0) return -1;
            break;
        }
        const unsigned char *t = p + sz - 4;
        const size_t isz = (size_t)t[0] | ((size_t)t[1] << 8) | ((size_t)t[2] << 16) | ((size_t)t[3] << 24);
        if (*isize_total + isz > out_cap) {
            if (*nm == 0) return -2;
            break;
        }
        *isize_total += isz;
        used += (size_t)sz;
        (*nm)++;
    }
    return (long)used;
}

static void *reader_main(void *arg)
{
    struct pipe_state *ps = (struct pipe_state *)arg;
    size_t carry = 0;
    unsigned char *carry_src = NULL;
    int eof_seen = 0;
    for (unsigned i = 0;; i++) {
        struct slot *sl = &ps->s[i % NSLOTS];
        wait_state(ps, sl, EMPTY);
        if (ps->failed) return NULL;
        if (carry) memmove(sl->in, carry_src, carry);      /* members left over from the previous slot */
        size_t have = carry;
        if (!eof_seen) {
            const double t0 = now_s();
            const size_t got = read_full(ps->fin, sl->in + carry, ps->in_cap - carry);
            g_t_read += now_s() - t0;
            have += got;
            eof_seen = got < ps->in_cap - carry;
        }
        carry = 0;
        sl->in_len = have;
        sl->members = 0;
        if (ps->decompress && have) {
            size_t nm, isz;
            const long used = whole_members(sl->in, have, ps->in_cap, ps->out_cap, eof_seen, &nm, &isz);
            if (used <= 0) {                               /* not a member, or one cut short by the end of the input */
                fprintf(stderr, used == -2 ? "a member larger than %zu MiB (compressed) / %zu MiB (payload) is not supported\n" : "not BGZF or corrupted\n",
                        ps->in_cap >> 20, ps->out_cap >> 20);
                fail(ps);
                return NULL;
            }
            sl->in_len = (size_t)used;
            sl->members = nm;
            carry = have - (size_t)used;
            carry_src = sl->in + used;
        }
        sl->last = eof_seen && carry == 0;
        set_state(ps, sl, FILLED);
        if (sl->last) return NULL;
    }
}

static void *writer_main(void *arg)
{
    struct pipe_state *ps = (struct pipe_state *)arg;
    for (unsigned i = 0;; i++) {
        struct slot *sl = &ps->s[i % NSLOTS];
        wait_state(ps, sl, DONE);
        if (ps->failed) return NULL;
        const double t0 = now_s();
        if (sl->out_len && fwrite(sl->out, 1, sl->out_len, ps->fout) != sl->out_len) { fail(ps); return NULL; }
        g_t_write += now_s() - t0;
        int last = sl->last;
        set_state(ps, sl, EMPTY);
        if (last) return NULL;
    }
}

/* ---- member index (--gzi): (compressed, uncompressed) start of every member, from the codec's own offsets ---- */
struct gzi_acc {
    uint64_t *caddr, *uaddr, *slot_off;
    size_t n, cap, slot_cap;
    uint64_t cbase, ubase;
};
static int gzi_add_slot(struct gzi_acc *g, size_t in_len, size_t out_len, uint32_t blk, int had_eof)
{
    const size_t nb = (in_len + blk - 1) / blk;
    if (g->n + nb > g->cap) {
        g->cap = (g->n + nb) * 2;
        g->caddr = (uint64_t *)realloc(g->caddr, g->cap * sizeof(uint64_t));
        g->uaddr = (uint64_t *)realloc(g->uaddr, g->cap * sizeof(uint64_t));
        if (!g->caddr || !g->uaddr) return -1;
    }
    for (size_t b = 0; b < nb; b++) {
        g->caddr[g->n] = g->cbase + g->slot_off[b];
        g->uaddr[g->n++] = g->ubase + (uint64_t)b * blk;
    }
    g->cbase += out_len - (had_eof ? B200BGZF_EOF_BYTES : 0);
    g->ubase += in_len;
    return 0;
}
static int gzi_write(const struct gzi_acc *g, const char *path)
{
    const size_t need = 8 + 16 * (g->n ? g->n - 1 : 0);
    unsigned char *buf = (unsigned char *)malloc(need);
    FILE *f = buf ? fopen(path, "wb") : NULL;
    int ok = f && b200bgzf_gzi_format(g->caddr, g->uaddr, g->n, buf, need) == need && fwrite(buf, 1, need, f) == need;
    if (f && fclose(f) != 0) ok = 0;
    free(buf);
    if (!ok) fprintf(stderr, "cannot write the index %s\n", path);
    return ok ? 0 : 1;
}

/* member starts of a stream by a header walk (the multi-GPU call reports no offsets) */
static size_t walk_member_offsets(const unsigned char *buf, size_t len, uint64_t *off, size_t cap)
{
    size_t n = 0, pos = 0;
    while (pos + 28 <= len && n < cap) {
        const size_t sz = ((size_t)buf[pos + 16] | ((size_t)buf[pos + 17] << 8)) + 1;
        off[n++] = pos;
        pos += sz;
    }
    return n;
}

/* The reader starts on stdin BEFORE the GPU context exists: creating a CUDA context takes 0.3 - 2 s, during which the first
 * slots fill.  Slots are plain page-aligned memory: pinning 400 MB costs 0.3 s, and the pipeline is bound by file I/O
 * (2 - 8 GB/s), not by the 10 GB/s at which the driver stages pageable buffers. */
static unsigned g_frame_flags;          /* B200BGZF_FRAME_MIGZ when run as `7migz` */
static int run_pipeline(int ndevices, int decompress, int level, uint32_t block, const char *gzi_path)
{
    b200bgzf_ctx *ctx = NULL;
    b200bgzf_multi *multi = NULL;
    struct gzi_acc gzi;
    memset(&gzi, 0, sizeof gzi);
    struct pipe_state ps;
    memset(&ps, 0, sizeof ps);
    pthread_mutex_init(&ps.mu, NULL);
    pthread_cond_init(&ps.cv, NULL);
    ps.fin = stdin;
    ps.fout = stdout;
    ps.decompress = decompress;
    if (decompress) {
        ps.in_cap = (size_t)16 << 20;        /* members are taken from here until their payloads fill ... */
        ps.out_cap = (size_t)96 << 20;       /* ... this much output (pinning memory costs ~0.4 ms per MiB: keep the slots modest) */
    } else {
        ps.in_cap = (size_t)SLOT_BLOCKS * block;
        ps.out_cap = b200bgzf_compress_bound(ps.in_cap, B200BGZF_BLOCK_SIZE) + 64 * B200BGZF_EOF_BYTES;   /* (the bound of the smaller block size is the larger one; room for the multi-GPU placement) */
    }
    const double ta = now_s();
    for (int i = 0; i < NSLOTS; i++) {
        void *a = NULL, *b = NULL;
        if (posix_memalign(&a, 4096, ps.in_cap) || posix_memalign(&b, 4096, ps.out_cap)) { fprintf(stderr, "out of memory\n"); return 1; }
        ps.s[i].in = (unsigned char *)a;
        ps.s[i].out = (unsigned char *)b;
        memset(b, 0, ps.out_cap);           /* fault the pages in now (the GPU context is not up yet anyway): a copy from the device
                                               into untouched pageable memory takes the driver's slow path */
    }
    g_t_alloc = now_s() - ta;
    if (gzi_path && !decompress) {
        gzi.slot_cap = (ps.in_cap + B200BGZF_BLOCK_SIZE - 1) / B200BGZF_BLOCK_SIZE;
        gzi.slot_off = (uint64_t *)malloc(gzi.slot_cap * sizeof(uint64_t));
        if (!gzi.slot_off) { fprintf(stderr, "out of memory\n"); return 1; }
    }
    pthread_t rd, wr;
    pthread_create(&rd, NULL, reader_main, &ps);
    pthread_create(&wr, NULL, writer_main, &ps);
    long units = 0;
    int ret = 0;
    {
        const double tc0 = now_s();
        const char *dev = getenv("B200BGZF_DEVICE");
        const int r = ndevices > 1 ? b200bgzf_multi_create(&multi, NULL, ndevices) : b200bgzf_create(&ctx, dev && *dev ? atoi(dev) : -1);
        g_t_create = now_s() - tc0;
        if (r != 0) {
            fprintf(stderr, "b200bgzf: cannot initialise the GPU codec: %s\n", b200bgzf_strerror(r));
            exit(1);                     /* (the reader may be blocked on stdin: do not wait for it) */
        }
    }
    for (unsigned i = 0; !ret; i++) {
        struct slot *sl = &ps.s[i % NSLOTS];
        wait_state(&ps, sl, FILLED);
        if (ps.failed) { ret = decompress ? -1 : 1; break; }
        sl->out_len = 0;
        const double tc = now_s();
        if (sl->in_len) {
            int r;
            if (decompress) {
                r = multi ? b200bgzf_multi_inflate_host(multi, sl->in, sl->in_len, sl->out, ps.out_cap, &sl->out_len, 0)
                          : b200bgzf_inflate_host(ctx, sl->in, sl->in_len, sl->out, ps.out_cap, &sl->out_len, 0);
                if (r != 0) { fprintf(stderr, "inflate %d\n", r); ret = 1; }
                units += (long)sl->members;
            } else {
                uint32_t used_block = block;
                const unsigned fl = (sl->last ? B200BGZF_APPEND_EOF : 0) | g_frame_flags;
                r = multi ? b200bgzf_multi_compress_host(multi, sl->in, sl->in_len, block, level, sl->out, ps.out_cap, &sl->out_len, fl)
                          : b200bgzf_compress_host_index(ctx, sl->in, sl->in_len, block, level, sl->out, ps.out_cap, &sl->out_len, fl, gzi.slot_off, gzi.slot_cap);
                if (r == B200BGZF_E_NOFIT && block > B200BGZF_BLOCK_SIZE) {
                    /* a 65536-byte payload that does not compress cannot fit a member: the reference's single-thread path
                     * shrinks the block and redoes it (7bgzf.c:135-147,256-262); here the slot is redone in 0xff00-byte
                     * blocks, which always fit */
                    used_block = B200BGZF_BLOCK_SIZE;
                    r = multi ? b200bgzf_multi_compress_host(multi, sl->in, sl->in_len, used_block, level, sl->out, ps.out_cap, &sl->out_len, fl)
                              : b200bgzf_compress_host_index(ctx, sl->in, sl->in_len, used_block, level, sl->out, ps.out_cap, &sl->out_len, fl, gzi.slot_off, gzi.slot_cap);
                    units += (long)((sl->in_len + B200BGZF_BLOCK_SIZE - 1) / B200BGZF_BLOCK_SIZE) - (long)((sl->in_len + block - 1) / block);
                }
                if (!r && multi && gzi.slot_off) walk_member_offsets(sl->out, sl->out_len, gzi.slot_off, gzi.slot_cap);
                if (r == B200BGZF_E_NOFIT) { fprintf(stderr, "libdeflate_deflate %d\n", 1); ret = 1; }
                else if (r != 0) { fprintf(stderr, "b200bgzf: %s (%s)\n", b200bgzf_strerror(r), b200bgzf_last_error(ctx)); ret = 1; }
                units += (long)((sl->in_len + block - 1) / block);
                if (!r && gzi.slot_off && gzi_add_slot(&gzi, sl->in_len, sl->out_len, used_block, sl->last)) { fprintf(stderr, "out of memory\n"); ret = 1; }
            }
        } else if (!decompress && sl->last && !g_frame_flags) {
            /* empty tail slot: still owe the EOF marker (7bgzf.c:283-289) */
            size_t n = 0;
            b200bgzf_compress_host(multi ? b200bgzf_multi_ctx(multi, 0) : ctx, NULL, 0, block, level, sl->out, ps.out_cap, &n, B200BGZF_APPEND_EOF);
            sl->out_len = n;
        }
        g_t_codec += now_s() - tc;
        if (ret) { fail(&ps); break; }
        fprintf(stderr, "%ld\r", units);
        int last = sl->last;
        set_state(&ps, sl, DONE);
        if (last) break;
    }
    pthread_join(rd, NULL);
    pthread_join(wr, NULL);
    if (ps.failed && !ret) ret = decompress ? -1 : 1;
    if (!ret && gzi.slot_off) ret = gzi_write(&gzi, gzi_path);
    free(gzi.caddr); free(gzi.uaddr); free(gzi.slot_off);
    if (!ret) fprintf(stderr, "%ld done.\n", units);
    if (getenv("B200BGZF_DEBUG"))
        fprintf(stderr, "stage seconds: slot alloc %.3f, context %.3f (reader already running), read %.3f, codec %.3f, write %.3f\n", g_t_alloc, g_t_create,
                g_t_read, g_t_codec, g_t_write);
    for (int i = 0; i < NSLOTS; i++) {
        free(ps.s[i].in);
        free(ps.s[i].out);
    }
    fflush(stdout);
    b200bgzf_destroy(ctx);
    b200bgzf_multi_destroy(multi);
    return ret;
}

/* ---- random access: the whole input in memory (a regular file is mapped: only the members a read touches are paged in) ---- */
struct input_map {
    unsigned char *p;
    size_t n, map_len;
    int mapped;
};
static int input_load(struct input_map *im)
{
    memset(im, 0, sizeof *im);
    struct stat st;
    const off_t pos = lseek(0, 0, SEEK_CUR);
    if (fstat(0, &st) == 0 && S_ISREG(st.st_mode) && pos >= 0 && st.st_size > pos) {
        void *m = mmap(NULL, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, 0, 0);
        if (m != MAP_FAILED) {
            im->p = (unsigned char *)m + pos;
            im->n = (size_t)(st.st_size - pos);
            im->map_len = (size_t)st.st_size;
            im->mapped = 1;
            return 0;
        }
    }
    size_t cap = (size_t)1 << 20;
    im->p = (unsigned char *)malloc(cap);
    for (;;) {
        if (!im->p) return -1;
        const ssize_t r = read(0, im->p + im->n, cap - im->n);
        if (r < 0) return -1;
        if (r == 0) return 0;
        im->n += (size_t)r;
        if (im->n == cap) im->p = (unsigned char *)realloc(im->p, cap *= 2);
    }
}
static void input_free(struct input_map *im)
{
    if (im->mapped) munmap(im->p - (im->map_len - im->n), im->map_len);
    else free(im->p);
}

/* the whole of an index file */
static int read_file(const char *path, unsigned char **buf, size_t *len)
{
    *buf = NULL;
    *len = 0;
    FILE *f = fopen(path, "rb");
    if (!f) { fprintf(stderr, "cannot read the index %s\n", path); return 1; }
    size_t cap = 4096;
    *buf = (unsigned char *)malloc(cap);
    for (size_t r; *buf && (r = fread(*buf + *len, 1, cap - *len, f)) > 0;)
        if ((*len += r) == cap) *buf = (unsigned char *)realloc(*buf, cap *= 2);
    fclose(f);
    if (!*buf) { fprintf(stderr, "out of memory\n"); return 1; }
    return 0;
}

/* (caddr, uaddr) of every member: from a .gzi, or by a header walk of the input */
static int load_index(const struct input_map *im, const char *gzi_path, uint64_t **c, uint64_t **u, size_t *n)
{
    *c = *u = NULL;
    *n = 0;
    unsigned char *buf = NULL;
    size_t len = 0;
    if (gzi_path && read_file(gzi_path, &buf, &len)) return 1;
    int r = gzi_path ? b200bgzf_gzi_parse(buf, len, NULL, NULL, 0, n) : b200bgzf_index_host(im->p, im->n, NULL, NULL, 0, n);
    if (r == 0 || r == B200BGZF_E_NOSPACE) {
        *c = (uint64_t *)malloc((*n + 1) * sizeof(uint64_t));
        *u = (uint64_t *)malloc((*n + 1) * sizeof(uint64_t));
        r = !*c || !*u ? B200BGZF_E_ARG
                       : gzi_path ? b200bgzf_gzi_parse(buf, len, *c, *u, *n, n) : b200bgzf_index_host(im->p, im->n, *c, *u, *n, n);
    }
    free(buf);
    if (r) fprintf(stderr, gzi_path ? "%s: not a .gzi index\n" : "not BGZF or corrupted\n", gzi_path);
    return r ? 1 : 0;
}

/* decoded size: start of the last member + its ISIZE */
static int stream_total(const struct input_map *im, const uint64_t *c, const uint64_t *u, size_t n, uint64_t *total)
{
    *total = 0;
    if (!n) return 0;
    uint64_t sz = 0;
    if (c[n - 1] >= im->n || !b200bgzf_member_header(im->p + c[n - 1], im->n - c[n - 1], &sz)) return 1;
    const unsigned char *t = im->p + c[n - 1] + sz - 4;
    *total = u[n - 1] + ((uint64_t)t[0] | ((uint64_t)t[1] << 8) | ((uint64_t)t[2] << 16) | ((uint64_t)t[3] << 24));
    return 0;
}

static int range_applet(uint64_t offset, uint64_t size, int have_size, const char *gzi_path)
{
    struct input_map im;
    if (input_load(&im)) { fprintf(stderr, "cannot read stdin\n"); return 1; }
    uint64_t *c = NULL, *u = NULL, total = 0;
    size_t n = 0;
    int ret = load_index(&im, gzi_path, &c, &u, &n);
    if (!ret && stream_total(&im, c, u, n, &total)) { fprintf(stderr, "not BGZF or corrupted\n"); ret = 1; }
    if (!ret && offset > total) { fprintf(stderr, "offset %llu is past the end of the data (%llu bytes)\n", (unsigned long long)offset, (unsigned long long)total); ret = 1; }
    if (!ret) {
        const uint64_t end = !have_size || size > total - offset ? total : offset + size;
        b200bgzf_range rg = { offset, end };
        unsigned char *out = (unsigned char *)malloc(end - offset + 1);
        b200bgzf_ctx *ctx = NULL;
        size_t got = 0;
        const char *dev = getenv("B200BGZF_DEVICE");
        int r = !out ? B200BGZF_E_ARG : b200bgzf_create(&ctx, dev && *dev ? atoi(dev) : -1);
        if (r) fprintf(stderr, "b200bgzf: cannot initialise the GPU codec: %s\n", b200bgzf_strerror(r));
        else if ((r = b200bgzf_inflate_ranges_host(ctx, im.p, im.n, c, u, n, &rg, 1, out, end - offset + 1, &got, NULL, 0)) != 0)
            fprintf(stderr, "inflate %d\n", r);
        if (!r && got && fwrite(out, 1, got, stdout) != got) r = 1;
        ret = r ? 1 : 0;
        b200bgzf_destroy(ctx);
        free(out);
    }
    free(c);
    free(u);
    input_free(&im);
    return ret;
}

/* bgzip -r: the .gzi of an existing stream (members that carry data; the first is implicit) */
static int reindex_applet(const char *gzi_path)
{
    struct input_map im;
    if (input_load(&im)) { fprintf(stderr, "cannot read stdin\n"); return 1; }
    uint64_t *c = NULL, *u = NULL, total = 0;
    size_t n = 0, k = 0;
    int ret = load_index(&im, NULL, &c, &u, &n);
    if (!ret && stream_total(&im, c, u, n, &total)) ret = 1;
    if (!ret) {
        for (size_t i = 0; i < n; i++)
            if ((i + 1 < n ? u[i + 1] : total) > u[i]) { c[k] = c[i]; u[k++] = u[i]; }
        struct gzi_acc g;
        memset(&g, 0, sizeof g);
        g.caddr = c;
        g.uaddr = u;
        g.n = k;
        ret = gzi_write(&g, gzi_path);
    }
    free(c);
    free(u);
    input_free(&im);
    return ret;
}

static b200bgzf_ctx *applet_ctx(void)
{
    b200bgzf_ctx *ctx = NULL;
    const char *dev = getenv("B200BGZF_DEVICE");
    const int r = b200bgzf_create(&ctx, dev && *dev ? atoi(dev) : -1);
    if (r) fprintf(stderr, "b200bgzf: cannot initialise the GPU codec: %s\n", b200bgzf_strerror(r));
    return r ? NULL : ctx;
}

/* 7gzip -d --offset=N [--size=M] --index=F: bytes [N, N+M) of a whole-stream gzip member (the decoded size is the index's
 * out_bytes field, include/b200bgzf.h) */
static int gzip_range_applet(uint64_t offset, uint64_t size, int have_size, const char *index_path)
{
    struct input_map im;
    if (input_load(&im)) { fprintf(stderr, "cannot read stdin\n"); return 1; }
    unsigned char *ix = NULL;
    size_t ixn = 0;
    uint64_t total = 0;
    int ret = read_file(index_path, &ix, &ixn);
    if (!ret && (ixn < 52 || memcmp(ix, "B2GZIX01", 8))) { fprintf(stderr, "%s: not a gzip index\n", index_path); ret = 1; }
    for (int k = 7; !ret && k >= 0; k--) total = total << 8 | ix[28 + k];
    if (!ret && offset > total) { fprintf(stderr, "offset %llu is past the end of the data (%llu bytes)\n", (unsigned long long)offset, (unsigned long long)total); ret = 1; }
    if (!ret) {
        const uint64_t end = !have_size || size > total - offset ? total : offset + size;
        b200bgzf_range rg = { offset, end };
        unsigned char *out = (unsigned char *)malloc(end - offset + 1);
        b200bgzf_ctx *ctx = out ? applet_ctx() : NULL;
        size_t got = 0;
        int r = ctx ? b200bgzf_gzip_inflate_ranges_host(ctx, im.p, im.n, ix, ixn, &rg, 1, out, end - offset + 1, &got, NULL, 0) : B200BGZF_E_ARG;
        if (r && ctx) fprintf(stderr, "%s: %s\n", index_path, b200bgzf_strerror(r));
        if (!r && got && fwrite(out, 1, got, stdout) != got) r = 1;
        ret = r ? 1 : 0;
        b200bgzf_destroy(ctx);
        free(out);
    }
    free(ix);
    input_free(&im);
    return ret;
}

/* 7gzip --reindex --index=F: the checkpoint index of the member on stdin (span 1 MiB) */
static int gzip_reindex_applet(const char *index_path)
{
    struct input_map im;
    if (input_load(&im)) { fprintf(stderr, "cannot read stdin\n"); return 1; }
    b200bgzf_ctx *ctx = applet_ctx();
    size_t cap = ((size_t)1 << 20) + im.n / 8, need = 0;   /* (a first guess: 32 KiB of window per MiB of output) */
    unsigned char *ix = (unsigned char *)malloc(cap);
    int r = !ctx || !ix ? B200BGZF_E_ARG : b200bgzf_gzip_index_host(ctx, im.p, im.n, 0, ix, cap, &need);
    if (r == B200BGZF_E_NOSPACE) {
        free(ix);
        ix = (unsigned char *)malloc(cap = need);
        r = ix ? b200bgzf_gzip_index_host(ctx, im.p, im.n, 0, ix, cap, &need) : B200BGZF_E_ARG;
    }
    if (r && ctx) fprintf(stderr, "cannot index this input: %s\n", b200bgzf_strerror(r));
    if (!r) {
        FILE *f = fopen(index_path, "wb");
        if (!f || fwrite(ix, 1, need, f) != need) r = 1;
        if (f && fclose(f)) r = 1;
        if (r) fprintf(stderr, "cannot write the index %s\n", index_path);
    }
    b200bgzf_destroy(ctx);
    free(ix);
    input_free(&im);
    return r ? 1 : 0;
}

int container_applet(const char *name, int kind, int decompress, int level, unsigned param, int ndevices, int nfiles, char **files);   /* applet_containers.c */

static const struct { const char *name; int kind; } k_personas[] = {
    { "7bgzf", 0 }, { "7migz", B200BGZF_CONTAINER_MIGZ }, { "7gzip", B200BGZF_CONTAINER_GZIP }, { "7gzinga", B200BGZF_CONTAINER_GZINGA },
    { "7dictzip", B200BGZF_CONTAINER_DICTZIP }, { "7razf", B200BGZF_CONTAINER_RAZF },
};

int main(int argc, char **argv)
{
    int levels[NFLAGS];
    int decompress = 0, nthreads = 1, bad = 0, ndevices = 1, migz = 0, bsize = 0, extreme = 0, kind = 0;
    int have_offset = 0, have_size = 0, reindex = 0;
    unsigned long long range_offset = 0, range_size = 0;
    unsigned piece_flags = 0;    /* 7gzip --independent: pieces without dictionary priming; 7migz --primed: with it */
    const char *gzi_path = NULL, *index_path = NULL, *persona = "7bgzf";
    memset(levels, 0, sizeof levels);
    /* allow `cielbox 7bgzf ...` style invocation.  As `7migz` (applet/7migz.c) with -b N <= 63 the same pipeline writes MiGz
     * members of N KiB (one member = one 64 KiB GPU slot); larger members (the reference's default is 512 KiB) and the
     * other containers (7gzip, 7gzinga, 7dictzip, 7razf) are made of several pieces: applet_containers.c */
    for (size_t k = 0; k < sizeof k_personas / sizeof k_personas[0]; k++)
        if (argc > 1 && !strcmp(argv[1], k_personas[k].name)) { argv++; argc--; break; }
    {
        const char *base = strrchr(argv[0], '/');
        base = base ? base + 1 : argv[0];
        for (size_t k = 0; k < sizeof k_personas / sizeof k_personas[0]; k++)
            if (!strcmp(base, k_personas[k].name)) { kind = k_personas[k].kind; persona = k_personas[k].name; }
        migz = kind == B200BGZF_CONTAINER_MIGZ;
    }

    static const struct option longopts[] = {
        { "stdout", no_argument, 0, 'c' },       { "zlib", optional_argument, 0, 'z' },
        { "miniz", optional_argument, 0, 'm' },  { "slz", optional_argument, 0, 's' },
        { "libdeflate", optional_argument, 0, 'l' }, { "7zip", optional_argument, 0, 'S' },
        { "zlibng", optional_argument, 0, 'n' }, { "cryptopp", optional_argument, 0, 'C' },
        { "igzip", optional_argument, 0, 'i' },  { "kzip", optional_argument, 0, 'K' },
        { "zopfli", required_argument, 0, 'Z' }, { "store", optional_argument, 0, 'T' },
        { "threads", required_argument, 0, '@' }, { "decompress", no_argument, 0, 'd' },
        { "help", no_argument, 0, 'h' },         { "gzi", required_argument, 0, 1000 },
        { "devices", required_argument, 0, 1001 },  { "bsize", required_argument, 0, 'b' },
        { "extreme", no_argument, 0, 'X' },      { "independent", no_argument, 0, 1002 },
        { "primed", no_argument, 0, 1003 },      { "offset", required_argument, 0, 1004 },
        { "size", required_argument, 0, 1005 },  { "reindex", no_argument, 0, 1006 },
        { "index", required_argument, 0, 1007 },
        { 0, 0, 0, 0 },
    };
    int opt;
    while ((opt = getopt_long(argc, argv, "cz::m::s::l::S::n::C::i::K::Z:T::@:dhb:X", longopts, NULL)) != -1) {
        if (opt == 'c') continue;
        if (opt == 'X') { extreme = 1; continue; }
        if (opt == 1002) { piece_flags |= B200BGZF_PARAM_INDEPENDENT; continue; }
        if (opt == 1003) { piece_flags |= B200BGZF_PARAM_PRIMED; continue; }
        if (opt == 'd') { decompress = 1; continue; }
        if (opt == '@') { nthreads = atoi(optarg); continue; }
        if (opt == 1000) { gzi_path = optarg; continue; }
        if (opt == 1001) { ndevices = atoi(optarg); if (ndevices < 1 || ndevices > 64) bad = 1; continue; }
        if (opt == 'b') { bsize = atoi(optarg); continue; }
        if (opt == 1004 || opt == 1005) {
            char *e = NULL;
            const unsigned long long v = strtoull(optarg, &e, 10);
            if (!*optarg || *e || *optarg == '-') bad = 1;
            if (opt == 1004) { range_offset = v; have_offset = 1; } else { range_size = v; have_size = 1; }
            continue;
        }
        if (opt == 1006) { reindex = 1; continue; }
        if (opt == 1007) { index_path = optarg; continue; }
        if (opt == 'h' || opt == '?') { bad = 1; continue; }
        for (size_t k = 0; k < NFLAGS; k++)
            if (k_flags[k].short_opt == opt)
                levels[k] = optarg ? (int)strtol(optarg, NULL, 10) : k_flags[k].default_level;
    }
    int chosen = -1, nchosen = 0, level_sum = 0;
    for (size_t k = 0; k < NFLAGS; k++)
        if (levels[k]) { chosen = (int)k; nchosen++; level_sum += levels[k]; }
    /* random access: 7bgzf -d --offset [--size] [--gzi], and --reindex --gzi; 7gzip the same with --index (required) */
    const int gz = kind == B200BGZF_CONTAINER_GZIP;
    if ((have_offset || have_size || reindex || index_path) && !bad) {
        if ((kind && !gz) || (gz ? !index_path || gzi_path : index_path != NULL) ||
            (reindex && (decompress || nchosen || have_offset || have_size || !(gz || gzi_path))) ||
            (!reindex && (!decompress || nchosen || !have_offset))) {
            usage(argv[0]);
            return 1;
        }
        if (isatty(fileno(stdin)) || (!reindex && isatty(fileno(stdout)))) {
            usage(argv[0]);
            return -1;
        }
        if (gz) return reindex ? gzip_reindex_applet(index_path) : gzip_range_applet(range_offset, range_size, have_size, index_path);
        return reindex ? reindex_applet(gzi_path) : range_applet(range_offset, range_size, have_size, gzi_path);
    }
    if (bad || (!decompress && nchosen != 1) || (decompress && nchosen != 0)) {
        usage(argv[0]);
        return 1;
    }
    struct timeval t0, t1;
    gettimeofday(&t0, NULL);
    if (migz && !bsize) bsize = 512;                               /* applet/7migz.c:327 */
    if (kind && !(migz && (decompress || (bsize <= 63 && !piece_flags)) && optind == argc)) {
        /* a container whose members span several pieces (or one that is read through its index) */
        int level = level_sum < 1 ? 1 : level_sum > 12 ? 12 : level_sum;
        if (!decompress) fprintf(stderr, "compression level = %d (%s)\n", level_sum, k_flags[chosen].label);
        if (migz && !decompress && (bsize < 1 || bsize > 4194303)) { fprintf(stderr, "7migz: -b %d: bad member size\n", bsize); return 1; }
        const unsigned param = (migz ? (unsigned)bsize : kind == B200BGZF_CONTAINER_DICTZIP && extreme ? B200BGZF_BLOCK_SIZE : 0u) | piece_flags;
        const int ret = container_applet(persona, kind, decompress, level, param, ndevices, argc - optind, argv + optind);
        gettimeofday(&t1, NULL);
        fprintf(stderr, "ellapsed time: %.6f sec\n", (t1.tv_sec + t1.tv_usec * 0.000001) - (t0.tv_sec + t0.tv_usec * 0.000001));
        return ret;
    }
    if (isatty(fileno(stdin)) || isatty(fileno(stdout))) {
        usage(argv[0]);
        return -1;
    }
    {
        struct stat st;
        g_in_regular = fstat(0, &st) == 0 && S_ISREG(st.st_mode);
        if (g_in_regular) g_in_pos = lseek(0, 0, SEEK_CUR);
        if (g_in_pos < 0) { g_in_regular = 0; g_in_pos = 0; }
    }
    int ret;
    if (decompress) {
        ret = run_pipeline(ndevices, 1, 0, 0, NULL);
    } else {
        int level = level_sum;
        fprintf(stderr, "compression level = %d (%s)\n", level_sum, k_flags[chosen].label);
        if (level < 1) level = 1;
        if (level > 12) level = 12;
        /* block size rule of the reference (7bgzf.c:141-147): 0x10000 with one thread, 0xff00 with -@N; the thread count has
         * no other meaning here (the GPU works on all blocks of a slot at once) */
        if (migz) g_frame_flags = B200BGZF_FRAME_MIGZ;
        ret = run_pipeline(ndevices, 0, level, migz ? (uint32_t)bsize * 1024u : nthreads == 1 ? B200BGZF_MAX_BLOCK_SIZE : B200BGZF_BLOCK_SIZE, gzi_path);
    }
    gettimeofday(&t1, NULL);
    fprintf(stderr, "ellapsed time: %.6f sec\n", (t1.tv_sec + t1.tv_usec * 0.000001) - (t0.tv_sec + t0.tv_usec * 0.000001));
    return ret;
}
