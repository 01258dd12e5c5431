/* TEST INFRASTRUCTURE ONLY.  csrc/mcb_trig.h against this machine's libm sinf and cosf.
 * Build: gcc -std=c11 -O2 -ffp-contract=off -pthread -o trig_exhaustive oracle/trig_exhaustive.c -lm
 * (tests/functions_common.py builds it that way into a temporary directory).
 *   exhaustive:  trig_exhaustive            every one of the 2^32 float bit patterns, both functions (about 45 s on 8 cores)
 *   strided:     trig_exhaustive 61         every 61st bit pattern
 *   random:      trig_exhaustive 1 N        N pseudo-random inputs plus the edge cases (signed zeros, subnormals,
 *                                           multiples of pi/2 and their neighbours, powers of two, the branch bounds
 *                                           of the algorithm, inf, NaN)
 * A mismatch is any difference of bits, except that two NaNs match.  It also counts finite results outside [-1, 1]
 * (mcb_interval.h encloses sin and cos of any interval by [-1, 1] on the strength of that count being 0). */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../marching-cube-for-implicit-surfaces_b200/csrc/mcb_trig.h"

typedef struct { uint64_t lo, hi, stride, n, bad_sin, bad_cos, out_of_range; } Job;

static float (*volatile libm_sin)(float) = sinf; /* called through a pointer: no constant folding, no builtin */
static float (*volatile libm_cos)(float) = cosf;

static int same(float a, float b) { return (a != a && b != b) || !memcmp(&a, &b, 4); }

static void check(Job* j, float x) {
    const float s = mcb_sinf(x), c = mcb_cosf(x);
    j->n++;
    if (!same(s, libm_sin(x))) {
        if (j->bad_sin < 3) printf("  sin x=%a (%08x) mcb=%a libm=%a\n", x, mcb_f2u(x), s, libm_sin(x));
        j->bad_sin++;
    }
    if (!same(c, libm_cos(x))) {
        if (j->bad_cos < 3) printf("  cos x=%a (%08x) mcb=%a libm=%a\n", x, mcb_f2u(x), c, libm_cos(x));
        j->bad_cos++;
    }
    if ((s == s && fabsf(s) <= INFINITY && !(s >= -1.0f && s <= 1.0f)) || (c == c && !(c >= -1.0f && c <= 1.0f)))
        j->out_of_range++;
}

static void* run(void* a) {
    Job* j = (Job*)a;
    for (uint64_t u = j->lo; u < j->hi; u += j->stride) check(j, mcb_u2f((uint32_t)u));
    return 0;
}

static uint64_t rng(uint64_t* s) { *s = *s * 6364136223846793005ull + 1442695040888963407ull; return *s >> 16; }

static int random_inputs(uint64_t n) {
    Job j;
    memset(&j, 0, sizeof j);
    const float edge[] = {0.0f, -0.0f, 1e-45f, -1e-45f, 1.17549435e-38f, 1.17549421e-38f, 0x1p-12f, 0x1.fffffep-13f,
                          0x1.921fb6p-1f, 0x1.921fb4p-1f, 120.0f, 0x1.dffffep6f, INFINITY, -INFINITY, NAN, -NAN,
                          3.40282347e38f, -3.40282347e38f, 1.0f, -1.0f};
    for (size_t i = 0; i < sizeof edge / sizeof edge[0]; i++) check(&j, edge[i]);
    for (int k = -149; k <= 127; k++) { /* powers of two and their neighbours */
        const float p = ldexpf(1.0f, k);
        for (int d = -2; d <= 2; d++) {
            const float v = mcb_u2f(mcb_f2u(p) + (uint32_t)d);
            check(&j, v);
            check(&j, -v);
        }
    }
    for (int m = -100000; m <= 100000; m++) { /* multiples of pi/2 (and of pi/4) in fp32, and their neighbours */
        const float v = (float)((double)m * 0x1.921fb54442d18p-1);
        for (int d = -3; d <= 3; d++) check(&j, mcb_u2f(mcb_f2u(v) + (uint32_t)d));
    }
    uint64_t st = 0x9E3779B97F4A7C15ull;
    for (uint64_t q = 0; q < n; q++) {
        uint32_t b = (uint32_t)rng(&st);
        if (q & 1) b = (b & 0x807fffffu) | ((100u + (uint32_t)(rng(&st) % 40u)) << 23); /* |x| in [2^-27, 2^12) */
        check(&j, mcb_u2f(b));
    }
    printf("random+edge inputs %llu mismatches_sin %llu mismatches_cos %llu out_of_range %llu\n", (unsigned long long)j.n,
           (unsigned long long)j.bad_sin, (unsigned long long)j.bad_cos, (unsigned long long)j.out_of_range);
    return j.bad_sin || j.bad_cos || j.out_of_range;
}

int main(int argc, char** argv) {
    enum { NT = 16 };
    if (argc > 2) return random_inputs(strtoull(argv[2], 0, 0));
    const uint64_t stride = argc > 1 ? strtoull(argv[1], 0, 0) : 1;
    pthread_t th[NT];
    Job jobs[NT];
    memset(jobs, 0, sizeof jobs);
    for (int t = 0; t < NT; t++) {
        jobs[t].lo = (1ull << 32) * t / NT; jobs[t].hi = (1ull << 32) * (t + 1) / NT; jobs[t].stride = stride;
        pthread_create(&th[t], 0, run, &jobs[t]);
    }
    uint64_t n = 0, bs = 0, bc = 0, oor = 0;
    for (int t = 0; t < NT; t++) {
        pthread_join(th[t], 0);
        n += jobs[t].n; bs += jobs[t].bad_sin; bc += jobs[t].bad_cos; oor += jobs[t].out_of_range;
    }
    printf("inputs %llu mismatches_sin %llu mismatches_cos %llu out_of_range %llu\n", (unsigned long long)n,
           (unsigned long long)bs, (unsigned long long)bc, (unsigned long long)oor);
    return bs || bc || oor ? 1 : 0;
}
