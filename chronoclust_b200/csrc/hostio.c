/*
 * hostio.c -- host-side writer of the per-cell output table (SURVEY 8f-2).
 *
 * The reference writes cluster_points_D{t}.csv with pandas (app.py:297-360: DataFrame.to_csv, one row per cell: id,
 * cluster_id, marker values).  At 1e6 cells x 12 markers that is ~10 s of single-threaded float formatting per timepoint
 * and it is most of the wall time of app.run once the clustering itself runs on the GPU.  This file produces the same
 * bytes with every host core: rows are cut into slabs, every slab is formatted by its own thread into its own buffer,
 * the buffers are written in order.
 *
 * Number formatting is Python's repr(float) -- what pandas' to_csv emits for float64 columns: the shortest decimal string
 * that round-trips, positional notation for 1e-4 <= |x| < 1e16 (with ".0" appended to integers), exponent notation
 * otherwise ("1e-05", "1.5e+16"); NaN becomes an empty field (na_rep=''), infinities "inf" / "-inf".  The shortest string
 * is found by trying 15, 16 and 17 significant digits (from 1 digit on for subnormals) ("%.{p}e" is correctly rounded in glibc) and checking the round trip
 * with strtod: if p digits suffice, the correctly rounded p-digit decimal is the shortest representation.
 *
 * It also holds the host side of the arcsinh transform, ccbio_arcsinh_host: the same csrc/asinh.h the kernels use, so
 * its output is the device's bit for bit.
 *
 * Plain C (gcc), pthreads; no CUDA here.  Built next to the CUDA library by chronoclust_b200/build.py, with
 * -ffp-contract=off (GNU C contracts a * b + c into an FMA by default where the target has one; asinh.h needs every
 * operation rounded on its own).
 */
#define _GNU_SOURCE
#include <errno.h>
#include <fcntl.h>
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include "asinh.h"

/* repr(v) into out (at least 32 bytes); returns the length */
static int fmt_repr(double v, char *out) {
    if (v != v) return 0; /* NaN -> empty field */
    if (isinf(v)) {
        const char *s = v > 0 ? "inf" : "-inf";
        const int n = (int)strlen(s);
        memcpy(out, s, (size_t)n);
        return n;
    }
    if (v == 0.0) {
        const char *s = signbit(v) ? "-0.0" : "0.0";
        const int n = (int)strlen(s);
        memcpy(out, s, (size_t)n);
        return n;
    }
    char buf[40];
    /* normal numbers carry >= 15.95 decimal digits, so the search starts at 15; subnormals carry fewer */
    int prec = fabs(v) < 2.2250738585072014e-308 ? 1 : 15;
    for (; prec <= 17; ++prec) {
        snprintf(buf, sizeof buf, "%.*e", prec - 1, v);
        if (prec == 17 || strtod(buf, NULL) == v) break;
    }
    /* buf = [-]d.ddddde[+-]XX[X] */
    const char *p = buf;
    int n = 0;
    if (*p == '-') out[n++] = *p++;
    char digits[20];
    int nd = 0;
    digits[nd++] = *p++;
    if (*p == '.') {
        ++p;
        while (*p && *p != 'e') digits[nd++] = *p++;
    }
    const int e10 = atoi(p + 1); /* p points at 'e' */
    while (nd > 1 && digits[nd - 1] == '0') --nd;
    const int decpt = e10 + 1; /* position of the decimal point relative to the first digit */
    if (decpt <= -4 || decpt > 16) { /* exponent notation: d[.ddd]e[+-]XX */
        out[n++] = digits[0];
        if (nd > 1) {
            out[n++] = '.';
            memcpy(out + n, digits + 1, (size_t)(nd - 1));
            n += nd - 1;
        }
        out[n++] = 'e';
        int e = decpt - 1;
        out[n++] = e < 0 ? '-' : '+';
        if (e < 0) e = -e;
        if (e >= 100) {
            out[n++] = (char)('0' + e / 100);
            e %= 100;
            out[n++] = (char)('0' + e / 10);
            out[n++] = (char)('0' + e % 10);
        } else {
            out[n++] = (char)('0' + e / 10);
            out[n++] = (char)('0' + e % 10);
        }
        return n;
    }
    if (decpt <= 0) { /* 0.000ddd */
        out[n++] = '0';
        out[n++] = '.';
        for (int i = 0; i < -decpt; ++i) out[n++] = '0';
        memcpy(out + n, digits, (size_t)nd);
        return n + nd;
    }
    if (decpt >= nd) { /* ddd000.0 */
        memcpy(out + n, digits, (size_t)nd);
        n += nd;
        for (int i = nd; i < decpt; ++i) out[n++] = '0';
        out[n++] = '.';
        out[n++] = '0';
        return n;
    }
    memcpy(out + n, digits, (size_t)decpt); /* dd.ddd */
    n += decpt;
    out[n++] = '.';
    memcpy(out + n, digits + decpt, (size_t)(nd - decpt));
    return n + nd - decpt;
}

static int fmt_i64(int64_t v, char *out) {
    char tmp[24];
    int n = 0, neg = v < 0;
    uint64_t u = neg ? (uint64_t)(-(v + 1)) + 1u : (uint64_t)v;
    do {
        tmp[n++] = (char)('0' + u % 10);
        u /= 10;
    } while (u);
    int m = 0;
    if (neg) out[m++] = '-';
    while (n) out[m++] = tmp[--n];
    return m;
}

typedef struct {
    int64_t r0, r1, id0;
    int32_t ncols;
    int64_t ld;
    const double *values;
    const int32_t *label_idx;
    const char *label_pool;
    const int64_t *label_off;
    char *buf;
    size_t len, cap;
    int err;
} slab_t;

static void *format_slab(void *arg) {
    slab_t *s = (slab_t *)arg;
    /* widest row: id (20) + label + ncols fields of <= 25 bytes + separators */
    size_t maxlab = 0;
    for (int64_t r = s->r0; r < s->r1; ++r) {
        const int32_t li = s->label_idx[r];
        const size_t l = (size_t)(s->label_off[li + 1] - s->label_off[li]);
        if (l > maxlab) maxlab = l;
    }
    const size_t rowmax = 24 + maxlab + (size_t)s->ncols * 26 + 4;
    s->cap = rowmax * (size_t)(s->r1 - s->r0) + 16;
    s->buf = (char *)malloc(s->cap);
    if (!s->buf) {
        s->err = ENOMEM;
        return NULL;
    }
    char *o = s->buf;
    for (int64_t r = s->r0; r < s->r1; ++r) {
        o += fmt_i64(s->id0 + r, o);
        *o++ = ',';
        const int32_t li = s->label_idx[r];
        const size_t l = (size_t)(s->label_off[li + 1] - s->label_off[li]);
        memcpy(o, s->label_pool + s->label_off[li], l);
        o += l;
        const double *row = s->values + r * s->ld;
        for (int c = 0; c < s->ncols; ++c) {
            *o++ = ',';
            o += fmt_repr(row[c], o);
        }
        *o++ = '\n';
    }
    s->len = (size_t)(o - s->buf);
    return NULL;
}

/* Writes `header` (one line, newline included) followed by n rows "id,label,v0,...,v{ncols-1}\n"; id = id0 + row.
 * values: [n][ld] doubles; label_idx [n] indexes the label table (label_pool + label_off [nlabels + 1]); labels must not
 * need CSV quoting.  nthreads <= 0: one per online core (at most 64).  Returns 0 or an errno value. */
int ccbio_write_points_csv(const char *path, const char *header, int64_t n, int32_t ncols, const double *values, int64_t ld,
                           int64_t id0, const int32_t *label_idx, const char *label_pool, const int64_t *label_off,
                           int32_t nthreads) {
    if (!path || !header || n < 0 || ncols < 0 || (n > 0 && (!values || !label_idx || !label_pool || !label_off)))
        return EINVAL;
    if (nthreads <= 0) nthreads = (int32_t)sysconf(_SC_NPROCESSORS_ONLN);
    if (nthreads > 64) nthreads = 64;
    if (nthreads < 1) nthreads = 1;
    const int64_t min_rows = 4096;
    int nslab = (int)((n + min_rows - 1) / min_rows);
    if (nslab > nthreads * 4) nslab = nthreads * 4; /* a few slabs per thread: the buffers stay small, the tail short */
    if (nslab < 1) nslab = 1;
    slab_t *slabs = (slab_t *)calloc((size_t)nslab, sizeof(slab_t));
    pthread_t *tids = (pthread_t *)calloc((size_t)nthreads, sizeof(pthread_t));
    if (!slabs || !tids) {
        free(slabs);
        free(tids);
        return ENOMEM;
    }
    for (int k = 0; k < nslab; ++k) {
        slab_t *s = &slabs[k];
        s->r0 = n * k / nslab;
        s->r1 = n * (k + 1) / nslab;
        s->id0 = id0;
        s->ncols = ncols;
        s->ld = ld;
        s->values = values;
        s->label_idx = label_idx;
        s->label_pool = label_pool;
        s->label_off = label_off;
    }
    int rc = 0;
    const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644);
    if (fd < 0) {
        rc = errno;
        goto done;
    }
    {
        const size_t hl = strlen(header);
        if (write(fd, header, hl) != (ssize_t)hl) rc = errno ? errno : EIO;
    }
    /* waves of nthreads slabs: format in parallel, then write the wave in order */
    for (int k0 = 0; k0 < nslab && !rc; k0 += nthreads) {
        const int k1 = k0 + nthreads < nslab ? k0 + nthreads : nslab;
        int started = 0;
        for (int k = k0; k < k1; ++k) {
            if (pthread_create(&tids[k - k0], NULL, format_slab, &slabs[k]) != 0) {
                format_slab(&slabs[k]); /* no thread available: do it here */
                tids[k - k0] = (pthread_t)0;
            } else {
                ++started;
            }
        }
        (void)started;
        for (int k = k0; k < k1; ++k)
            if (tids[k - k0]) pthread_join(tids[k - k0], NULL);
        for (int k = k0; k < k1; ++k) {
            slab_t *s = &slabs[k];
            if (s->err && !rc) rc = s->err;
            size_t off = 0;
            while (!rc && off < s->len) {
                const ssize_t w = write(fd, s->buf + off, s->len - off);
                if (w < 0) {
                    if (errno == EINTR) continue;
                    rc = errno;
                } else {
                    off += (size_t)w;
                }
            }
            free(s->buf);
            s->buf = NULL;
        }
    }
    if (close(fd) != 0 && !rc) rc = errno;
done:
    for (int k = 0; k < nslab; ++k) free(slabs[k].buf);
    free(slabs);
    free(tids);
    return rc;
}

typedef struct {
    const void *X;
    int32_t dtype, D;
    int64_t r0, r1, ld;
    const double *cofactor;
    double *out;
} asinh_slab_t;

static void *asinh_slab(void *arg) {
    const asinh_slab_t *s = (const asinh_slab_t *)arg;
    for (int64_t r = s->r0; r < s->r1; ++r) {
        double *o = s->out + r * s->D;
        for (int d = 0; d < s->D; ++d) {
            double x = s->dtype == 1 ? (double)((const float *)s->X)[r * s->ld + d] : ((const double *)s->X)[r * s->ld + d];
            if (s->cofactor[d] != 0.0) x = ccb_asinh(x / s->cofactor[d]);
            o[d] = x;
        }
    }
    return NULL;
}

/* out [N][D] (float64, contiguous) = X [N][ld] (dtype 0: float64, 1: float32) widened to double, and every column d with
 * cofactor[d] != 0 transformed to ccb_asinh(x / cofactor[d]) -- ccb_arcsinh's values, bit for bit.  Cofactors are
 * checked by the caller.  nthreads <= 0: one per online core (at most 64).  Returns 0 or an errno value. */
int ccbio_arcsinh_host(const void *X, int32_t dtype, int64_t N, int64_t ld, int32_t D, const double *cofactor, double *out,
                       int32_t nthreads) {
    if (N < 0 || D < 0 || ld < D || (dtype != 0 && dtype != 1) || (N > 0 && (!X || !cofactor || !out))) return EINVAL;
    if (nthreads <= 0) nthreads = (int32_t)sysconf(_SC_NPROCESSORS_ONLN);
    if (nthreads > 64) nthreads = 64;
    if (nthreads < 1) nthreads = 1;
    if ((int64_t)nthreads > (N + 4095) / 4096) nthreads = (int32_t)((N + 4095) / 4096); /* >= 4096 rows a thread */
    if (nthreads < 1) nthreads = 1;
    asinh_slab_t slabs[64];
    pthread_t tids[64];
    for (int k = 0; k < nthreads; ++k) {
        asinh_slab_t *s = &slabs[k];
        s->X = X, s->dtype = dtype, s->D = D, s->ld = ld, s->cofactor = cofactor, s->out = out;
        s->r0 = N * k / nthreads, s->r1 = N * (k + 1) / nthreads;
        if (k == 0 || pthread_create(&tids[k], NULL, asinh_slab, s) != 0) {
            asinh_slab(s); /* the first slab, or no thread available: do it here */
            tids[k] = (pthread_t)0;
        }
    }
    for (int k = 1; k < nthreads; ++k)
        if (tids[k]) pthread_join(tids[k], NULL);
    return 0;
}

/* repr(v) for tests: writes into out (>= 32 bytes), returns the length */
int ccbio_repr(double v, char *out) { return fmt_repr(v, out); }
