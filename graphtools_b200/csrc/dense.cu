// K5: dense exact graph.  Tiled all-pairs float64 distances with the alpha-decay kernel,
// thresholding and the symmetrisation fused per output tile (S_ij depends only on d_ij, bw_i, bw_j,
// so no transpose is needed), row sums accumulated on the fly, then one scaling sweep for P.
//
// Replaces TraditionalGraph.build_kernel / build_kernel_to_data (reference graphtools/graphs.py
// :1546-1609, :1651-1677: scipy pdist/squareform/cdist + numpy partition/power/exp) and the dense
// branches of symmetrize_kernel / apply_anisotropy / normalize (base.py:557-592, :645).
// Distances are float64 direct differences of the inputs as given -- float32 rows or float64 rows (PCA output,
// float64 user data), template T -- which is what scipy's pdist / cdist compute.  Metrics: euclidean, cosine,
// cityblock, sqeuclidean (correlation is the cosine branch on row-centred float64 rows, prepared by the caller as
// scipy does).  Row sums are NOT accumulated here (a floating-point atomic per tile would make the degree vector
// depend on the tile order): gtb_dense_rowsum makes one deterministic pass afterwards.
#include "common.cuh"
#include "gtb200.h"

namespace {

constexpr int DT = 64;    // output tile edge
constexpr int DK = 16;    // feature chunk

enum { DENSE_DIST = 0, DENSE_KERNEL = 1, DENSE_KERNEL_SYM = 2 };

__device__ __forceinline__ double sym_dense(int mode, double theta, double a, double b) {
  if (mode == 0) return (a + b) / 2;
  if (mode == 1) return a * b;
  if (mode == 2) return theta * fmin(a, b) + (1 - theta) * fmax(a, b);
  return a;
}

// out[i][j] for i in query rows (Xq), j in reference rows (Xr).
template <typename T>
__global__ void __launch_bounds__(256) dense_kernel(const T* __restrict__ Xq, int64_t nq,
                                                    const T* __restrict__ Xr, int64_t nr, int d, int what,
                                                    int metric, const double* __restrict__ bw_q, const double* __restrict__ bw_r,
                                                    double decay, double thresh, double rfac, int symm,
                                                    double theta, double* __restrict__ out,
                                                    double* __restrict__ rowsum) {
  __shared__ double qs[DK][DT + 1];
  __shared__ double rs[DK][DT + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 x 16 threads, 4 x 4 outputs each
  const int64_t i0 = (int64_t)blockIdx.y * DT, j0 = (int64_t)blockIdx.x * DT;
  double acc[4][4];
  double qn[4] = {0.0, 0.0, 0.0, 0.0}, rn[4] = {0.0, 0.0, 0.0, 0.0};   // squared row norms (cosine metric)
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;

  for (int k0 = 0; k0 < d; k0 += DK) {
    // cooperative load: 64 rows x 16 features for both operands (thread -> 4 elements each)
    for (int e = threadIdx.x; e < DT * DK; e += 256) {
      int r = e / DK, k = e % DK;
      int64_t gi = i0 + r, gj = j0 + r;
      qs[k][r] = (gi < nq && k0 + k < d) ? (double)Xq[gi * d + k0 + k] : 0.0;
      rs[k][r] = (gj < nr && k0 + k < d) ? (double)Xr[gj * d + k0 + k] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < DK; ++k) {
      double qv[4], rv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) { qv[a] = qs[k][ty * 4 + a]; rv[a] = rs[k][tx * 4 + a]; }
      if (metric == 1) {
        // cosine: accumulate the dot products and the squared norms (scipy cdist / pdist "cosine")
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          qn[a] = fma(qv[a], qv[a], qn[a]);
          rn[a] = fma(rv[a], rv[a], rn[a]);
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b] = fma(qv[a], rv[b], acc[a][b]);
        }
      } else if (metric == 2) {
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b] += fabs(qv[a] - rv[b]);
      } else {
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            double df = qv[a] - rv[b];
            acc[a][b] = fma(df, df, acc[a][b]);
          }
      }
    }
    __syncthreads();
  }

#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int64_t i = i0 + ty * 4 + a;
    double rsum = 0.0;
    if (i < nq) {
      const double bwi = (what != DENSE_DIST) ? bw_q[i] : 1.0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int64_t j = j0 + tx * 4 + b;
        if (j >= nr) continue;
        double dist;
        if (metric == 1) {
          // an all-zero row has no direction: NaN, as in scipy (the kernel below maps it to 1 like the reference)
          double c = (qn[a] == 0.0 || rn[b] == 0.0) ? NAN : acc[a][b] / (sqrt(qn[a]) * sqrt(rn[b]));
          if (fabs(c) > 1.0) c = copysign(1.0, c);
          dist = 1.0 - c;
        } else if (metric == 2 || metric == 3) {
          dist = acc[a][b];
        } else {
          dist = sqrt(acc[a][b]);
        }
        double v;
        if (what == DENSE_DIST) {
          v = dist;
        } else {
          // pairs beyond the kernel support radius bw * (-ln thresh)^(1/decay) are zero: skip pow/exp
          // (the 1e-9 guard keeps every value that could round to >= thresh on the exact path); a NaN distance or
          // bandwidth passes the test and gtb_affinity turns it into 1, np.where(isnan(K), 1, K) in the reference
          v = 0.0;
          if (!(dist > bwi * rfac)) {
            v = gtb_affinity(dist, bwi, decay);
            if (v < thresh) v = 0.0;
          }
          if (what == DENSE_KERNEL_SYM) {
            double vr = 0.0;
            const double bwj = bw_r[j];
            if (!(dist > bwj * rfac)) {
              vr = gtb_affinity(dist, bwj, decay);
              if (vr < thresh) vr = 0.0;
            }
            v = sym_dense(symm, theta, v, vr);
          }
        }
        out[i * nr + j] = v;
        rsum += fabs(v);
      }
    }
    (void)rsum; (void)rowsum;
  }
}

// out = in / rowsum (rows with zero sum untouched) -- sklearn normalize(K, 'l1') dense branch
__global__ void dense_row_scale_kernel(const double* __restrict__ in, const double* __restrict__ rowsum, int64_t nq,
                                       int64_t nr, double* __restrict__ out) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nq * nr) return;
  double s = rowsum[e / nr];
  double v = in[e];
  out[e] = (s != 0.0) ? v / s : v;
}

// K_ij /= (deg_i deg_j)^alpha, new row sums accumulated (dense apply_anisotropy, base.py:589-591)
__global__ void dense_anisotropy_kernel(double* __restrict__ K, const double* __restrict__ deg, double alpha,
                                        int64_t n, double* __restrict__ newsum) {
  const int lane = threadIdx.x & 31;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const double di = deg[row];
  double s = 0.0;
  for (int64_t j = lane; j < n; j += 32) {
    double v = K[row * n + j] / pow(di * deg[j], alpha);
    K[row * n + j] = v;
    s += fabs(v);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if (lane == 0) newsum[row] = s;
}

__global__ void dense_rowsum_kernel(const double* __restrict__ K, int64_t nq, int64_t nr, double* __restrict__ sum) {
  const int lane = threadIdx.x & 31;
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= nq) return;
  double s = 0.0;
  for (int64_t j = lane; j < nr; j += 32) s += fabs(K[row * nr + j]);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if (lane == 0) sum[row] = s;
}

}  // namespace

extern "C" int gtb_dense_kernel(const void* Xq, int64_t nq, const void* Xr, int64_t nr, int d, int x_is_f64, int what,
                                int metric, const double* bw_q, const double* bw_r, double decay, double thresh, int symm,
                                double theta, double* out, double* rowsum, void* stream) {
  GTB_CHECK_ARG(nq > 0 && nr > 0 && d > 0, "empty input");
  GTB_CHECK_ARG(what >= 0 && what <= 2, "bad mode");
  GTB_CHECK_ARG(metric >= 0 && metric <= 3, "metric must be 0 (euclidean), 1 (cosine), 2 (cityblock) or 3 (sqeuclidean)");
  GTB_CHECK_ARG(what == 0 || bw_q != nullptr, "bandwidth required");
  GTB_CHECK_ARG(what != 2 || (bw_r != nullptr && nq == nr), "symmetric mode needs a square problem");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((unsigned)gtb_cdiv(nr, DT), (unsigned)gtb_cdiv(nq, DT));
  // support radius factor; +inf when nothing is thresholded away (thresh <= 0) or in distance mode
  double rfac = INFINITY;
  if (what != DENSE_DIST && thresh > 0 && thresh < 1 && decay > 0) rfac = pow(-log(thresh), 1.0 / decay) * (1.0 + 1e-9);
  if (x_is_f64)
    dense_kernel<double><<<grid, 256, 0, st>>>((const double*)Xq, nq, (const double*)Xr, nr, d, what, metric, bw_q, bw_r,
                                               decay, thresh, rfac, symm, theta, out, nullptr);
  else
    dense_kernel<float><<<grid, 256, 0, st>>>((const float*)Xq, nq, (const float*)Xr, nr, d, what, metric, bw_q, bw_r,
                                              decay, thresh, rfac, symm, theta, out, nullptr);
  GTB_CHECK_LAUNCH();
  if (rowsum) {
    dense_rowsum_kernel<<<(unsigned)gtb_cdiv(nq * 32, 256), 256, 0, st>>>(out, nq, nr, rowsum);
    GTB_CHECK_LAUNCH();
  }
  return GTB_OK;
}

extern "C" int gtb_dense_row_scale(const double* in, const double* rowsum, int64_t nq, int64_t nr, double* out,
                                   void* stream) {
  dense_row_scale_kernel<<<(unsigned)gtb_cdiv(nq * nr, 256), 256, 0, (cudaStream_t)stream>>>(in, rowsum, nq, nr, out);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_dense_anisotropy(double* K, const double* deg, double alpha, int64_t n, double* newsum,
                                    void* stream) {
  dense_anisotropy_kernel<<<(unsigned)gtb_cdiv(n * 32, 256), 256, 0, (cudaStream_t)stream>>>(K, deg, alpha, n, newsum);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}

extern "C" int gtb_dense_rowsum(const double* K, int64_t nq, int64_t nr, double* sum, void* stream) {
  dense_rowsum_kernel<<<(unsigned)gtb_cdiv(nq * 32, 256), 256, 0, (cudaStream_t)stream>>>(K, nq, nr, sum);
  GTB_CHECK_LAUNCH();
  return GTB_OK;
}
