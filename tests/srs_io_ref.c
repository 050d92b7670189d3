/* tests/srs_io_ref.c — CPU reference for the compressed G1 codec (TEST INFRASTRUCTURE, never linked into the product).
 *
 * G1Affine::from_bytes as upstream (dusk-bls12_381 0.8) states it and csrc/verify.cu restates it on the host: flag checks,
 * x < p, y = (x³ + 4)^((p+1)/4), y² = x³ + 4, the root the flag asks for, and the subgroup check r·P = O — deliberately the
 * plain definition, not the endomorphism test the GPU codec (csrc/g1_codec.cuh) uses, so the two are independent.
 * Status codes are PB200_G1_* of include/pb200.h.  Points are split over `threads` pthreads.
 *
 * The field and curve arithmetic is the CPU checker's own: oracle/oracle.c is compiled into this translation unit
 * unchanged (its static helpers — fp_*, g1p_add, g1p_mul_u — become visible here), so the decoder shares no code with the
 * library.  Build: gcc -O3 -march=x86-64-v3 -madx -fPIC -shared tests/srs_io_ref.c -lpthread (tests/srs_io_ref.py does). */
#include "../oracle/oracle.c"

enum { REF_OK = 0, REF_BAD_FLAGS = 1, REF_X_RANGE = 2, REF_NOT_ON_CURVE = 3, REF_NOT_IN_SUBGROUP = 4, REF_IDENTITY = 5 };

static const uint64_t SQRT_EXP[6] = {0xee7fbfffffffeaabull, 0x07aaffffac54ffffull, 0xd9cc34a83dac3d89ull,
                                     0xd91dd2e13ce144afull, 0x92c6e9ed90d2eb35ull, 0x0680447a8e5ff9a6ull}; /* (p + 1)/4 */

/* 2·y ≥ p for a canonical y */
static int larger_root(const fp_t *yc) {
    fp_t d;
    uint64_t carry = fp_raw_add(&d, yc, yc);
    return carry || fp_geq(&d, &fp_MOD);
}
static int ref_decode(const uint8_t *b, fp_t *x_out, fp_t *y_out) {
    if (!(b[0] & 0x80)) return REF_BAD_FLAGS;
    if (b[0] & 0x40) {
        if (b[0] != 0xc0) return REF_BAD_FLAGS;
        for (int i = 1; i < 48; i++)
            if (b[i]) return REF_BAD_FLAGS;
        return REF_IDENTITY;
    }
    fp_t raw;
    for (int i = 0; i < 6; i++) {
        raw.l[i] = 0;
        for (int k = 7; k >= 0; k--) {
            uint8_t byte = b[47 - (8 * i + k)];
            if (8 * i + k == 47) byte &= 0x1f;
            raw.l[i] = (raw.l[i] << 8) | byte;
        }
    }
    if (fp_geq(&raw, &fp_MOD)) return REF_X_RANGE;
    fp_t x, t, rhs, four, y;
    fp_to_mont(&x, &raw);
    fp_sqr(&t, &x);
    fp_mul(&rhs, &t, &x);
    fp_from_u64(&four, 4);
    fp_add(&rhs, &rhs, &four);
    fp_pow(&y, &rhs, SQRT_EXP, 6);
    fp_sqr(&t, &y);
    if (!fp_eq(&t, &rhs)) return REF_NOT_ON_CURVE;
    fp_from_mont(&t, &y);
    if (larger_root(&t) != !!(b[0] & 0x20)) fp_neg(&y, &y);
    g1a_t a;
    a.x = x;
    a.y = y;
    a.inf = 0;
    g1p_t p, q;
    g1p_from_affine(&p, &a);
    g1p_mul_u(&q, &p, FR_MODULUS, 4);
    if (!g1p_is_identity(&q)) return REF_NOT_IN_SUBGROUP;
    *x_out = x;
    *y_out = y;
    return REF_OK;
}
static void ref_encode(const uint64_t *xy_mont, uint8_t *out) {
    fp_t x, y;
    memcpy(x.l, xy_mont, 48);
    memcpy(y.l, xy_mont + 6, 48);
    fp_from_mont(&x, &x);
    fp_from_mont(&y, &y);
    for (int i = 0; i < 48; i++) out[47 - i] = (uint8_t)(x.l[i / 8] >> (8 * (i % 8)));
    out[0] |= 0x80 | (larger_root(&y) ? 0x20 : 0);
}

typedef struct {
    const uint8_t *bytes;
    uint64_t *xy;
    uint8_t *status;
    size_t lo, hi;
    int encode;
} ref_job_t;
static void *ref_worker(void *arg) {
    const ref_job_t *J = (const ref_job_t *)arg;
    for (size_t i = J->lo; i < J->hi; i++) {
        if (J->encode) {
            ref_encode(J->xy + 12 * i, (uint8_t *)J->bytes + 48 * i);
            continue;
        }
        fp_t x, y;
        const int st = ref_decode(J->bytes + 48 * i, &x, &y);
        J->status[i] = (uint8_t)st;
        if (st == REF_OK) {
            memcpy(J->xy + 12 * i, x.l, 48);
            memcpy(J->xy + 12 * i + 6, y.l, 48);
        } else {
            memset(J->xy + 12 * i, 0, 96);
        }
    }
    return NULL;
}
static void ref_run(const uint8_t *bytes, uint64_t *xy, uint8_t *status, size_t n, int threads, int encode) {
    orc_init();
    if (threads < 1) threads = 1;
    if ((size_t)threads > n) threads = n ? (int)n : 1;
    pthread_t *th = malloc(threads * sizeof(pthread_t));
    ref_job_t *jobs = malloc(threads * sizeof(ref_job_t));
    for (int t = 0; t < threads; t++) {
        jobs[t] = (ref_job_t){bytes, xy, status, n * t / threads, n * (t + 1) / threads, encode};
        pthread_create(&th[t], NULL, ref_worker, &jobs[t]);
    }
    for (int t = 0; t < threads; t++) pthread_join(th[t], NULL);
    free(th);
    free(jobs);
}

/* n 48-byte encodings → status per point and the packed affine point (x ‖ y, 12 u64 Montgomery; zero when invalid). */
ORC_API void orc_g1_from_bytes_checked(const uint8_t *bytes, size_t n, uint64_t *out_xy_mont, uint8_t *status, int threads) {
    ref_run(bytes, out_xy_mont, status, n, threads, 0);
}
/* n packed affine points (12 u64 Montgomery each) → 48-byte encodings. */
ORC_API void orc_g1_to_bytes(const uint64_t *xy_mont, size_t n, uint8_t *out, int threads) {
    ref_run(out, (uint64_t *)xy_mont, NULL, n, threads, 1);
}
