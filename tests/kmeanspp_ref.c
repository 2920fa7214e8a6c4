/* kmeanspp_ref.c — the reference's k-means++ seeding loop, sequential, for the tests of nk_index_kmeanspp.
 * initCentroidsKMeansPlusPlus (pkg/gpu/kmeans.go:364-427) with the random numbers injected: rand.Intn(n) -> first,
 * the c-th rand.Float64() -> draws[c-1].  squaredEuclidean (kmeans.go:430-454): float32 differences, float64 squares,
 * four partial sums.  Built with -ffp-contract=off so a square and its sum round separately, as in Go on amd64. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static double sq_euclid64(const float *a, const float *b, uint32_t n) {
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    uint32_t i = 0;
    for (; i + 4 <= n; i += 4) {
        const double d0 = (double)(a[i] - b[i]), d1 = (double)(a[i + 1] - b[i + 1]);
        const double d2 = (double)(a[i + 2] - b[i + 2]), d3 = (double)(a[i + 3] - b[i + 3]);
        s0 += d0 * d0;
        s1 += d1 * d1;
        s2 += d2 * d2;
        s3 += d3 * d3;
    }
    for (; i < n; ++i) {
        const double d = (double)(a[i] - b[i]);
        s0 += d * d;
    }
    return s0 + s1 + s2 + s3;
}

/* centroids_out [K x dim], rows_out [K]; returns 0, or -1 when out of memory */
int ref_kmeanspp(const float *rows, uint64_t n, uint32_t dim, uint32_t K, uint64_t first, const double *draws, float *centroids_out,
                 uint32_t *rows_out) {
    double *mind = (double *)malloc(n * sizeof(double));
    if (!mind) return -1;
    memcpy(centroids_out, rows + first * dim, dim * sizeof(float));
    rows_out[0] = (uint32_t)first;
    for (uint64_t i = 0; i < n; ++i) mind[i] = sq_euclid64(rows + i * dim, centroids_out, dim);
    for (uint32_t c = 1; c < K; ++c) {
        double total = 0.0;
        for (uint64_t i = 0; i < n; ++i) total += mind[i];
        const double target = draws[c - 1] * total;
        double cum = 0.0;
        uint64_t sel = n - 1;
        for (uint64_t i = 0; i < n; ++i) {
            cum += mind[i];
            if (cum >= target) {
                sel = i;
                break;
            }
        }
        float *cen = centroids_out + (size_t)c * dim;
        memcpy(cen, rows + sel * dim, dim * sizeof(float));
        rows_out[c] = (uint32_t)sel;
        for (uint64_t i = 0; i < n; ++i) {
            const double d = sq_euclid64(rows + i * dim, cen, dim);
            if (d < mind[i]) mind[i] = d;
        }
    }
    free(mind);
    return 0;
}
