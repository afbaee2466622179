/* bgzf_gzip_route.h — between the GZIP container reader (host/containers.c) and the parallel whole-stream inflate
 * (b200bgzf_api.cu, bgzf_gzip.cu).  Not exported. */
#ifndef BGZF_GZIP_ROUTE_H
#define BGZF_GZIP_ROUTE_H
#include <stddef.h>
#include <stdint.h>

#include "../../include/b200bgzf.h"

#define BGZF_GZIP_FALLBACK 100   /* neither parallel route (flush points, searched block starts) takes the member: decode it on one warp */

#ifdef __cplusplus
extern "C" {
#endif
/* RFC 1952 header: its length (0: not a gzip member / cut short) and where the extra field lies */
size_t bgzf_gz_header(const uint8_t *p, size_t avail, size_t *xoff, size_t *xlen);
/* one member spanning in[0, in_bytes) with a header of hdr_len bytes: the outcome, or BGZF_GZIP_FALLBACK */
int bgzf_gzip_inflate_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t hdr_len, void *out, size_t out_cap,
                           size_t *out_bytes, unsigned flags);
#ifdef __cplusplus
}
#endif
#endif
