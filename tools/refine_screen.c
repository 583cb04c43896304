/* The error of the reference's float NXC chain against the exact correlation, for the screen of the uint8 subpixel refine
 * (libbicos_b200/csrc/refine.cu, the note above refine_kernel). Used by tests/test_refine_screen.py through ctypes.
 *
 * Build: gcc -std=c11 -O2 -ffp-contract=off -shared -fPIC (fmaf through libm, no contraction: the chain is the
 * reference's operation for operation, like oracle/bicos_oracle.c).
 */
#include <math.h>
#include <stdint.h>

/* include/impl/cpu/agree.hpp:28-51 without the min-variance test: sequential float mean, fmaf chains. var1 is the
 * float variance of the right stack. */
static float nxcorr_f32(const uint8_t* p0, const uint8_t* p1, int n, float* var1_out) {
    float mean0 = 0.f, mean1 = 0.f;
    for (int i = 0; i < n; ++i) {
        mean0 += (float)p0[i];
        mean1 += (float)p1[i];
    }
    mean0 /= (float)n;
    mean1 /= (float)n;
    float covar = 0.f, var0 = 0.f, var1 = 0.f;
    for (int i = 0; i < n; ++i) {
        const float diff0 = (float)p0[i] - mean0, diff1 = (float)p1[i] - mean1;
        covar = fmaf(diff0, diff1, covar);
        var0 = fmaf(diff0, diff0, var0);
        var1 = fmaf(diff1, diff1, var1);
    }
    *var1_out = var1;
    return covar / sqrtf(var0 * var1);
}

static uint64_t next(uint64_t* s) { /* xorshift64* */
    uint64_t x = *s;
    x ^= x >> 12;
    x ^= x << 25;
    x ^= x >> 27;
    *s = x;
    return x * 0x2545F4914F6CDD1DULL;
}

static int below(uint64_t* s, int k) {
    return (int)((next(s) >> 33) % (uint64_t)k);
}

/* Stacks of one kind:
 *  0  uniform random
 *  1  nearly constant: a base value and a few entries one or two away (tiny variances, means far from 0)
 *  2  right stack of exactly two values, one of them once: var_n = n - 1, the smallest nonzero variance
 *  3  anti-correlated: right = 255 - left + small noise
 *  4  strongly correlated: right = left + small noise, clipped
 *  5  ties: few left values, and right values swapped between images of equal left value, which keeps the exact
 *     correlation and changes the order of the float chains
 */
static void draw(uint64_t* s, int kind, int n, uint8_t* l, uint8_t* v) {
    switch (kind) {
    case 1: {
        const int b0 = below(s, 256), b1 = below(s, 256);
        for (int t = 0; t < n; ++t) {
            l[t] = (uint8_t)b0;
            v[t] = (uint8_t)b1;
        }
        const int k = 1 + below(s, 3);
        for (int i = 0; i < k; ++i) {
            int a = l[below(s, n)] + below(s, 5) - 2, b = v[below(s, n)] + below(s, 5) - 2;
            l[below(s, n)] = (uint8_t)(a < 0 ? 0 : a > 255 ? 255 : a);
            v[below(s, n)] = (uint8_t)(b < 0 ? 0 : b > 255 ? 255 : b);
        }
        break;
    }
    case 2: {
        const int b = below(s, 255);
        for (int t = 0; t < n; ++t) {
            l[t] = (uint8_t)below(s, 256);
            v[t] = (uint8_t)b;
        }
        v[below(s, n)] = (uint8_t)(b + 1);
        break;
    }
    case 3:
    case 4:
        for (int t = 0; t < n; ++t) {
            l[t] = (uint8_t)below(s, 256);
            int x = (kind == 3 ? 255 - l[t] : l[t]) + below(s, 7) - 3;
            v[t] = (uint8_t)(x < 0 ? 0 : x > 255 ? 255 : x);
        }
        break;
    case 5:
        for (int t = 0; t < n; ++t) {
            l[t] = (uint8_t)below(s, 4); /* few left values: equal pairs everywhere */
            v[t] = (uint8_t)below(s, 256);
        }
        for (int i = 0; i < 4; ++i) {
            const int a = below(s, n), b = below(s, n);
            if (l[a] == l[b]) {
                const uint8_t x = v[a];
                v[a] = v[b];
                v[b] = x;
            }
        }
        break;
    default:
        for (int t = 0; t < n; ++t) {
            l[t] = (uint8_t)below(s, 256);
            v[t] = (uint8_t)below(s, 256);
        }
    }
}

/* Over `count` stacks of `kind`: the largest |float NXC - exact rho| and the largest |float var1 / (var1_n / n) - 1|,
 * both in units of 2^-24, over the stacks whose two variances are nonzero. Returns the number of such stacks. */
long rs_worst_error(int n, long count, uint64_t seed, int kind, double* nxc_err, double* var_err) {
    uint8_t l[128], v[128];
    uint64_t s = seed * 0x9E3779B97F4A7C15ULL + 1;
    double worst = 0.0, worst_var = 0.0;
    long used = 0;
    for (long i = 0; i < count; ++i) {
        draw(&s, kind, n, l, v);
        long sl = 0, sv = 0, sll = 0, svv = 0, slv = 0;
        for (int t = 0; t < n; ++t) {
            sl += l[t];
            sv += v[t];
            sll += l[t] * l[t];
            svv += v[t] * v[t];
            slv += l[t] * v[t];
        }
        const long var0 = n * sll - sl * sl, var1 = n * svv - sv * sv, cov = n * slv - sl * sv;
        if (var0 == 0 || var1 == 0)
            continue;
        ++used;
        const double rho = (double)cov / sqrt((double)var0 * (double)var1);
        float fv1;
        const float f = nxcorr_f32(l, v, n, &fv1);
        const double e = fabs((double)f - rho) * 16777216.0;
        const double ev = fabs((double)fv1 / ((double)var1 / n) - 1.0) * 16777216.0;
        if (e > worst)
            worst = e;
        if (ev > worst_var)
            worst_var = ev;
    }
    *nxc_err = worst;
    *var_err = worst_var;
    return used;
}
