// Multi-start expansion (tg_multistart_expand): B problems x K seeded starts -> B * K rows, start-major within a
// problem (row b * K + k), for an ordinary solve of all rows; tg_multistart_select (tg_kernels_eval.inc) keeps the best.
//
// The start model.  Start 0 is x0[b] bit for bit.  Start k > 0 moves two things:
//   * the interior control points j = 3 .. N-4 of every coordinate c (the three at each end enter the terminal
//     waypoint rows and stay put) by  spread * l * s_kc(j),  l = |P_{N-1} - P_0| of x0[b].  The profile s_kc is zero at
//     j = 2 and j = N-3 and interpolates linearly between TG_MS_KNOTS knot values spaced evenly in between; knot q of
//     (k, c) is splitmix64(splitmix64(seed) + (k * 4 + c) * 8 + q) mapped to [-1, 1) through its top 53 bits;
//   * the scale factor alpha, multiplied by tg_ms_alpha_factor(k): 1, 1/2, 2, 3/4, 3/2, 5/8, 5/4, 3, repeating with
//     period 8 (all exact binary fractions).
// Waypoint scalars and intermediate times are copied: every start stays inside the solver's bounds.  Nothing depends
// on b, so equal problems get equal starts at any batch position.  Only correctly rounded operations (+ - x / and
// sqrt, no contraction), so a numpy restatement reproduces every start bit for bit (tests/test_multistart.py).
#include <cuda_runtime.h>
#include <stdint.h>
#include "tg_spec.h"
#include "tg_shape.h"

#define TG_MS_KNOTS 3

namespace {

__device__ __forceinline__ uint64_t tg_splitmix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// knot value q (0 .. TG_MS_KNOTS + 1; the two end knots are 0) of coordinate c of start k, in [-1, 1)
__device__ __forceinline__ double tg_ms_knot(uint64_t seed, int k, int c, int q)
{
    if (q <= 0 || q > TG_MS_KNOTS) return 0.0;
    const uint64_t h = tg_splitmix64(tg_splitmix64(seed) + ((uint64_t)k * 4 + (uint64_t)c) * 8 + (uint64_t)q);
    return __dsub_rn(__dmul_rn((double)(h >> 11), 0x1p-52), 1.0);
}

__device__ __forceinline__ double tg_ms_alpha_factor(int k)
{
    switch (k & 7) {
    case 1: return 0.5;
    case 2: return 2.0;
    case 3: return 0.75;
    case 4: return 1.5;
    case 5: return 0.625;
    case 6: return 1.25;
    case 7: return 3.0;
    default: return 1.0;
    }
}

// one thread per element of x_out, then of par_out
__global__ void __launch_bounds__(256) tg_multistart_expand_kernel(const TgLayout L, int B, int K, const double *__restrict__ par,
                                                                   const double *__restrict__ x0, uint64_t seed, double spread,
                                                                   double *__restrict__ par_out, double *__restrict__ x_out)
{
    const size_t rows = (size_t)B * K, nx = rows * L.n, total = nx + rows * L.P;
    const int N = L.N, W = N - 5;           // profile window: j = 2 .. N-3
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        if (e >= nx) {
            const size_t q = e - nx, row = q / L.P;
            par_out[q] = par[(row / K) * L.P + q % L.P];
            continue;
        }
        const size_t row = e / L.n, b = row / K;
        const int i = (int)(e % L.n), k = (int)(row % K);
        const double *xb = x0 + b * L.n;
        double v = xb[i];
        if (k > 0 && i == L.ia) {
            v = __dmul_rn(v, tg_ms_alpha_factor(k));
        } else if (k > 0 && i < L.ia) {
            const int c = i / N, j = i % N;
            if (j >= 3 && j <= N - 4) {
                double l2 = 0;
                for (int cc = 0; cc < L.d; cc++) {
                    const double dl = __dsub_rn(xb[cc * N + N - 1], xb[cc * N]);
                    l2 = cc == 0 ? __dmul_rn(dl, dl) : __dadd_rn(l2, __dmul_rn(dl, dl));
                }
                const double len = __dsqrt_rn(l2);
                const int t = (j - 2) * (TG_MS_KNOTS + 1), q = t / W;
                const double w = __ddiv_rn((double)(t % W), (double)W);
                const double v0 = tg_ms_knot(seed, k, c, q), v1 = tg_ms_knot(seed, k, c, q + 1);
                const double s = __dadd_rn(v0, __dmul_rn(w, __dsub_rn(v1, v0)));
                v = __dadd_rn(v, __dmul_rn(__dmul_rn(spread, len), s));
            }
        }
        x_out[e] = v;
    }
}

}  // namespace

cudaError_t tg_launch_multistart_expand(const TgLayout &L, int B, int K, const double *par, const double *x0,
                                        unsigned long long seed, double spread, double *par_out, double *x_out,
                                        int sm_count, cudaStream_t st)
{
    const size_t total = (size_t)B * K * (L.n + L.P);
    size_t grid = (total + 255) / 256;
    if (grid > (size_t)sm_count * 16) grid = (size_t)sm_count * 16;
    tg_multistart_expand_kernel<<<(unsigned)grid, 256, 0, st>>>(L, B, K, par, x0, (uint64_t)seed, spread, par_out, x_out);
    return cudaGetLastError();
}
