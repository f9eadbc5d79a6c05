// K8: randomized truncated SVD of the URM (PureSVD).  Replaces sklearn.utils.extmath.randomized_svd as
// MatrixFactorization/PureSVDRecommender.py:36-55 calls it.
//
// Layout: every dense block is row-major fp32 with a leading dimension `ld` (a multiple of 4) and `l <= ld` active
// columns; the padding columns are kept at zero, so the SpMM can stream whole float4 rows.
//   - csr_spmm_kernel: Y = A X, one group of g lanes per output row, each lane owning float4 column slices; no atomics.
//   - orthonormalisation: shifted CholeskyQR3 -- fp64 Gram with per-tile partials summed in a fixed order, fp64
//     Cholesky + triangular inverse in one CTA, Q = Y R^-1 by a tall x small fp64-accumulated product.  A pivot at or
//     below tau * (largest diagonal) in an unshifted pass (or a non-positive pivot in any pass) marks the column
//     deficient: it is refilled with Philox Gaussians and the pass is repeated.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <math.h>
#include <algorithm>
#include <utility>
#include <vector>

#include "common.cuh"

namespace b200 {
namespace rsvd {

constexpr int MAX_L = 512;
constexpr double TAU = 1e-10;  // relative pivot below which an unshifted pass declares a column deficient

// ---- Y[r, :] = sum_j val[j] X[idx[j], :]  (nq = ld / 4 float4 columns; C float4 slices per lane) ----------------
template <int C>
__global__ void __launch_bounds__(256) csr_spmm_kernel(long long n_rows, const int* __restrict__ ptr, const int* __restrict__ idx,
                                                       const float* __restrict__ val, const float4* __restrict__ X, int nq, int g,
                                                       float4* __restrict__ Y) {
  const int lane = threadIdx.x & 31, lg = threadIdx.x & (g - 1);
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / g;
  if (row >= n_rows) return;  // whole groups leave together
  const unsigned mask = g == 32 ? 0xffffffffu : (((1u << g) - 1u) << (lane & ~(g - 1)));
  float4 acc[C];
#pragma unroll
  for (int t = 0; t < C; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int b = ptr[row], e = ptr[row + 1];
  for (int j0 = b; j0 < e; j0 += g) {
    const int mine = j0 + lg;
    const int my_c = mine < e ? __ldg(idx + mine) : 0;
    const float my_v = mine < e ? __ldg(val + mine) : 0.f;
    const int cnt = min(g, e - j0);
#pragma unroll 4
    for (int s = 0; s < cnt; ++s) {
      const int c = __shfl_sync(mask, my_c, s, g);
      const float v = __shfl_sync(mask, my_v, s, g);
      const float4* xr = X + (size_t)c * nq;
#pragma unroll
      for (int t = 0; t < C; ++t) {
        const int q = lg + t * g;
        if (q < nq) {
          const float4 x = __ldg(xr + q);
          acc[t].x = fmaf(v, x.x, acc[t].x);
          acc[t].y = fmaf(v, x.y, acc[t].y);
          acc[t].z = fmaf(v, x.z, acc[t].z);
          acc[t].w = fmaf(v, x.w, acc[t].w);
        }
      }
    }
  }
  float4* yr = Y + (size_t)row * nq;
#pragma unroll
  for (int t = 0; t < C; ++t) {
    const int q = lg + t * g;
    if (q < nq) yr[q] = acc[t];
  }
}

// ---- CSR transpose: row id of every stored entry, then a stable radix sort by column --------------------------------
__global__ void entry_rows_kernel(long long n_rows, long long nnz, const int* __restrict__ ptr, int* rows, int* pos, int* col_cnt,
                                  const int* __restrict__ idx) {
  const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (j >= nnz) return;
  long long lo = 0, hi = n_rows;  // last row r with ptr[r] <= j
  while (hi - lo > 1) {
    const long long mid = (lo + hi) >> 1;
    if (ptr[mid] <= j) lo = mid; else hi = mid;
  }
  rows[j] = (int)lo;
  pos[j] = (int)j;
  atomicAdd(col_cnt + idx[j], 1);
}

__global__ void gather_transpose_kernel(long long nnz, const int* __restrict__ perm, const int* __restrict__ rows,
                                        const float* __restrict__ val, int* t_idx, float* t_val) {
  const long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  const int j = perm[p];
  t_idx[p] = rows[j];
  t_val[p] = val[j];
}

// ---- P[s, i, j] = sum over the rows of chunk s of X[r, i] Y[r, j]  (fp64; 64 x 64 output tile, 4 x 4 per thread) -----
__global__ void __launch_bounds__(256) xty_partial_kernel(long long n, int la, int lb, const float* __restrict__ X, int ldx,
                                                          const float* __restrict__ Y, int ldy, long long chunk, double* P) {
  __shared__ double xs[32][64], ys[32][64];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int i0 = blockIdx.x * 64, j0 = blockIdx.y * 64;
  const long long rb = blockIdx.z * chunk, re = min(n, rb + chunk);
  double acc[4][4] = {};
  for (long long r0 = rb; r0 < re; r0 += 32) {
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int e = tid + 256 * t, rr = e >> 6, cc = e & 63;
      const long long r = r0 + rr;
      xs[rr][cc] = (r < re && i0 + cc < la) ? (double)X[r * ldx + i0 + cc] : 0.0;
      ys[rr][cc] = (r < re && j0 + cc < lb) ? (double)Y[r * ldy + j0 + cc] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { a[u] = xs[k][ty + 16 * u]; b[u] = ys[k][tx + 16 * u]; }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fma(a[u], b[v], acc[u][v]);
    }
    __syncthreads();
  }
  double* Ps = P + (size_t)blockIdx.z * la * lb;
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
      if (i < la && j < lb) Ps[(size_t)i * lb + j] = acc[u][v];
    }
}

// fixed-order sum of the partials: the Gram is bit-identical from run to run
__global__ void sum_partials_kernel(int n_out, int n_parts, const double* __restrict__ P, double* G) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_out) return;
  double s = 0.0;
  for (int p = 0; p < n_parts; ++p) s += P[(size_t)p * n_out + o];
  G[o] = s;
}

// ---- Cholesky G (+ shift I) = R^T R and R^-1, fp64, one CTA of 512 threads --------------------------------------------
// M: the l x l working matrix (shared memory when it fits, else global); on return Rinv (global) holds R^-1 (upper).
// bad[k] = 1 for a deficient column k (its row of R is set to e_k); info[0] = number of deficient columns, dinfo[0] = the
// largest diagonal of G.
__global__ void __launch_bounds__(512) chol_inv_kernel(int l, double* G, double shift_coef, double tau, int use_smem, double* Rinv_g,
                                                        int* bad, int* info, double* dinfo) {
  extern __shared__ double sm[];
  __shared__ double s_red[32];
  __shared__ double s_piv;
  __shared__ int s_bad_cnt;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int ll = l * l;
  double* R = use_smem ? sm : G;
  double* Ri = use_smem ? sm + ll : Rinv_g;
  if (use_smem)
    for (int e = tid; e < ll; e += nt) R[e] = G[e];
  if (tid == 0) s_bad_cnt = 0;
  __syncthreads();
  // largest diagonal and trace (shift = shift_coef * ||Y||_F^2)
  double dmax = 0.0, tr = 0.0;
  for (int i = tid; i < l; i += nt) { const double d = R[i * l + i]; dmax = fmax(dmax, d); tr += d; }
  for (int o = 16; o; o >>= 1) { dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o)); tr += __shfl_xor_sync(0xffffffffu, tr, o); }
  if ((tid & 31) == 0) s_red[tid >> 5] = dmax;
  __syncthreads();
  if (tid == 0) { double m = 0.0; for (int w = 0; w < nt / 32; ++w) m = fmax(m, s_red[w]); s_piv = m; }
  __syncthreads();
  dmax = s_piv;
  __syncthreads();
  if ((tid & 31) == 0) s_red[tid >> 5] = tr;
  __syncthreads();
  if (tid == 0) { double t = 0.0; for (int w = 0; w < nt / 32; ++w) t += s_red[w]; s_piv = t; }
  __syncthreads();
  const double shift = shift_coef * s_piv;
  for (int i = tid; i < l; i += nt) R[i * l + i] += shift;
  __syncthreads();
  for (int k = 0; k < l; ++k) {
    if (tid == 0) {
      const double d = R[k * l + k];
      const bool deficient = !(d > tau * dmax) || !(d > 0.0) || !isfinite(d);
      bad[k] = deficient;
      if (deficient) ++s_bad_cnt;
      s_piv = deficient ? 0.0 : sqrt(d);
    }
    __syncthreads();
    const double piv = s_piv;
    if (piv == 0.0) {
      for (int j = k + tid; j < l; j += nt) R[k * l + j] = j == k ? 1.0 : 0.0;
      __syncthreads();
      continue;
    }
    const double inv = 1.0 / piv;
    for (int j = k + 1 + tid; j < l; j += nt) R[k * l + j] *= inv;
    __syncthreads();
    if (tid == 0) R[k * l + k] = piv;
    const int m = l - k - 1;
    for (int e = tid; e < m * m; e += nt) {
      const int i = k + 1 + e / m, j = k + 1 + e % m;
      if (j >= i) R[i * l + j] -= R[k * l + i] * R[k * l + j];
    }
    __syncthreads();
  }
  // R^-1 by rows from the bottom: Ri[i, j] = (delta_ij - sum_{i<t<=j} R[i, t] Ri[t, j]) / R[i, i], one warp per j
  for (int e = tid; e < ll; e += nt) Ri[e] = 0.0;
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
  for (int i = l - 1; i >= 0; --i) {
    const double rii = R[i * l + i];
    for (int j = i + warp; j < l; j += nw) {
      double s = 0.0;
      for (int t = i + 1 + lane; t <= j; t += 32) s += R[i * l + t] * Ri[t * l + j];
      for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) Ri[i * l + j] = ((i == j ? 1.0 : 0.0) - s) / rii;
    }
    __syncthreads();
  }
  if (use_smem)
    for (int e = tid; e < ll; e += nt) Rinv_g[e] = Ri[e];
  if (tid == 0) { info[0] = s_bad_cnt; dinfo[0] = dmax; }
}

// ---- C[r, j] = sum_{i < la} X[r, i] S[i, j]  (X fp32, S fp64, fp64 accumulation, C fp32; 64 x 64 tile, 4 x 4 per thread) -
__global__ void __launch_bounds__(256) tall_small_kernel(long long n, int la, int lc, const float* __restrict__ X, int ldx,
                                                         const double* __restrict__ S, int lds, float* __restrict__ Cm, int ldc) {
  __shared__ double xs[32][65], ss[32][64];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long r0 = (long long)blockIdx.x * 64;
  const int c0 = blockIdx.y * 64;
  double acc[4][4] = {};
  for (int i0 = 0; i0 < la; i0 += 32) {
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const int e = tid + 256 * t;
      const int rr = e >> 5, ii = e & 31;  // X tile: 64 rows x 32 columns, read along the row
      const long long r = r0 + rr;
      xs[ii][rr] = (r < n && i0 + ii < la) ? (double)X[r * ldx + i0 + ii] : 0.0;
      const int si = e >> 6, sc = e & 63;  // S tile: 32 rows x 64 columns
      ss[si][sc] = (i0 + si < la && c0 + sc < lc) ? S[(size_t)(i0 + si) * lds + c0 + sc] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { a[u] = xs[k][ty + 16 * u]; b[u] = ss[k][tx + 16 * u]; }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = fma(a[u], b[v], acc[u][v]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const long long r = r0 + ty + 16 * u;
    if (r >= n) continue;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int c = c0 + tx + 16 * v;
      if (c < lc) Cm[r * ldc + c] = (float)acc[u][v];
    }
  }
}

// deficient columns -> Gaussian columns of norm ~ sqrt(largest Gram diagonal) (Philox, key = (seed, attempt))
__global__ void refill_kernel(long long n, int l, int ld, float* Y, const int* __restrict__ bad, const double* __restrict__ dinfo,
                              unsigned seed, unsigned attempt) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= n * l) return;
  const long long r = e / l;
  const int c = (int)(e % l);
  if (!bad[c]) return;
  const double dm = dinfo[0];
  const float scale = (float)(dm > 0.0 ? sqrt(dm / (double)n) : 1.0 / sqrt((double)n));
  const uint4 w = philox((unsigned long long)e, 0u, seed, attempt);
  const float u1 = ((w.x >> 8) + 1) * (1.0f / 16777216.0f), u2 = (w.y >> 8) * (1.0f / 16777216.0f);
  Y[r * ld + c] = scale * sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// ---- svd_flip: per column of the user-side factor, the first row of largest |value| and its sign ---------------------
__global__ void colmax_partial_kernel(long long n, int k, const float* __restrict__ U, int ldu, long long chunk, float* pmax,
                                      long long* parg) {
  const long long rb = blockIdx.y * chunk, re = min(n, rb + chunk);
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < k; j += gridDim.x * blockDim.x) {
    float best = -1.f;
    long long arg = rb;
    for (long long r = rb; r < re; ++r) {
      const float a = fabsf(U[r * ldu + j]);
      if (a > best) { best = a; arg = r; }
    }
    pmax[(size_t)blockIdx.y * k + j] = best;
    parg[(size_t)blockIdx.y * k + j] = arg;
  }
}

__global__ void colsign_kernel(int k, int n_parts, const float* __restrict__ pmax, const long long* __restrict__ parg,
                               const float* __restrict__ U, int ldu, float* sign) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= k) return;
  float best = -1.f;
  long long arg = 0;
  for (int p = 0; p < n_parts; ++p)
    if (pmax[(size_t)p * k + j] > best) { best = pmax[(size_t)p * k + j]; arg = parg[(size_t)p * k + j]; }
  sign[j] = U[arg * ldu + j] < 0.f ? -1.f : 1.f;
}

__global__ void scale_cols_kernel(long long n, int k, float* F, const float* __restrict__ sign, const float* __restrict__ sigma) {
  const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (e >= n * k) return;
  const int j = (int)(e % k);
  F[e] *= sigma ? sign[j] * sigma[j] : sign[j];
}

// ---- host side ---------------------------------------------------------------------------------------------------------
void spmm(long long n_rows, const int* ptr, const int* idx, const float* val, const float* X, int ld, float* Y, cudaStream_t st) {
  const int nq = ld / 4;
  int g = 1;
  while (g < nq && g < 32) g <<= 1;
  const int C = (nq + g - 1) / g;
  if (n_rows == 0) return;
  const unsigned grid = div_up(n_rows * g, 256);
  const float4* X4 = reinterpret_cast<const float4*>(X);
  float4* Y4 = reinterpret_cast<float4*>(Y);
  switch (C) {
    case 1: csr_spmm_kernel<1><<<grid, 256, 0, st>>>(n_rows, ptr, idx, val, X4, nq, g, Y4); break;
    case 2: csr_spmm_kernel<2><<<grid, 256, 0, st>>>(n_rows, ptr, idx, val, X4, nq, g, Y4); break;
    case 3: csr_spmm_kernel<3><<<grid, 256, 0, st>>>(n_rows, ptr, idx, val, X4, nq, g, Y4); break;
    default: csr_spmm_kernel<4><<<grid, 256, 0, st>>>(n_rows, ptr, idx, val, X4, nq, g, Y4); break;
  }
  B200_CUDA(cudaGetLastError());
  count_launch();
}

void tall_small(long long n, int la, int lc, const float* X, int ldx, const double* S, int lds, float* Cm, int ldc, cudaStream_t st) {
  if (n == 0) return;
  tall_small_kernel<<<dim3(div_up(n, 64), div_up(lc, 64)), 256, 0, st>>>(n, la, lc, X, ldx, S, lds, Cm, ldc);
  B200_CUDA(cudaGetLastError());
  count_launch();
}

// Scratch of the l x l steps, sized once per call.
struct Work {
  int l = 0, n_parts = 0;
  long long chunk = 0;
  DevBuf<double> partials, G, Rinv, dinfo;
  DevBuf<int> bad, info;
  Work(long long n_max, int l_) : l(l_) {
    const int tiles = (int)(div_up(l, 64) * div_up(l, 64));
    long long parts = std::max(1LL, (2LL * sm_count() + tiles - 1) / tiles);
    parts = std::min(parts, std::max(1LL, (long long)div_up(n_max, 256)));
    parts = std::min(parts, std::max(1LL, (8LL << 20) / ((long long)l * l)));
    n_parts = (int)parts;
    partials.alloc((size_t)n_parts * l * l);
    G.alloc((size_t)l * l);
    Rinv.alloc((size_t)l * l);
    dinfo.alloc(1);
    bad.alloc((size_t)l);
    info.alloc(1);
  }
  // G = X^T Y over n rows (l x l, fp64, fixed summation order)
  void xty(long long n, const float* X, const float* Y, int ld, cudaStream_t st) {
    const long long ch = std::max(32LL, ((n + n_parts - 1) / n_parts + 31) / 32 * 32);
    const int parts = (int)std::max(1LL, (n + ch - 1) / ch);
    if (n == 0) {
      B200_CUDA(cudaMemsetAsync(G.get(), 0, sizeof(double) * l * l, st));
      return;
    }
    xty_partial_kernel<<<dim3(div_up(l, 64), div_up(l, 64), parts), 256, 0, st>>>(n, l, l, X, ld, Y, ld, ch, partials.get());
    B200_CUDA(cudaGetLastError());
    sum_partials_kernel<<<div_up((long long)l * l, 256), 256, 0, st>>>(l * l, parts, partials.get(), G.get());
    B200_CUDA(cudaGetLastError());
    count_launch(2);
  }
};

// In-place orthonormalisation of the n x l block Y (ld columns stored); tmp: another n x ld buffer with zero padding.
// Returns the number of deficient columns refilled.
int orthonormalize(Work& w, long long n, int l, int ld, float* Y, float* tmp, unsigned seed, cudaStream_t st) {
  const size_t smem = (size_t)2 * l * l * sizeof(double);
  const int use_smem = smem <= 200 * 1024;
  if (use_smem) B200_CUDA(cudaFuncSetAttribute(chol_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // Fukaya et al. (2020) shift for an fp64 Gram: 11 (n l + l (l + 1)) u ||Y||_F^2
  const double shift_coef = 11.0 * ((double)n * l + (double)l * (l + 1)) * 1.1102230246251565e-16;
  float* cur = Y;
  float* other = tmp;
  int breakdowns = 0, attempts = 0, clean = 0;
  bool shifted = true;
  while (clean < 2) {
    w.xty(n, cur, cur, ld, st);
    chol_inv_kernel<<<1, 512, use_smem ? smem : 0, st>>>(l, w.G.get(), shifted ? shift_coef : 0.0, shifted ? 0.0 : TAU, use_smem,
                                                          w.Rinv.get(), w.bad.get(), w.info.get(), w.dinfo.get());
    B200_CUDA(cudaGetLastError());
    count_launch();
    int n_bad = 0;
    B200_CUDA(cudaMemcpyAsync(&n_bad, w.info.get(), sizeof(int), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    if (n_bad > 0) {
      B200_REQUIRE(++attempts <= 8, "orthonormalize: %d columns still deficient after 8 refills", n_bad);
      refill_kernel<<<div_up(n * l, 256), 256, 0, st>>>(n, l, ld, cur, w.bad.get(), w.dinfo.get(), seed, (unsigned)attempts);
      B200_CUDA(cudaGetLastError());
      count_launch();
      breakdowns += n_bad;
      continue;
    }
    tall_small(n, l, l, cur, ld, w.Rinv.get(), l, other, ld, st);
    std::swap(cur, other);
    if (shifted) shifted = false; else ++clean;
  }
  if (cur != Y) B200_CUDA(cudaMemcpyAsync(Y, cur, sizeof(float) * (size_t)n * ld, cudaMemcpyDeviceToDevice, st));
  return breakdowns;
}

// phase timer: CUDA events around each phase, summed when the caller asks for the totals
struct Timer {
  bool on;
  cudaStream_t st;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[2];
  Timer(bool on_, cudaStream_t s) : on(on_), st(s) {}
  ~Timer() {
    for (auto& v : ev)
      for (auto& p : v) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  }
  void begin(int phase) {
    if (!on) return;
    cudaEvent_t a, b;
    B200_CUDA(cudaEventCreate(&a));
    B200_CUDA(cudaEventCreate(&b));
    ev[phase].push_back({a, b});
    B200_CUDA(cudaEventRecord(a, st));
  }
  void end(int phase) {
    if (on) B200_CUDA(cudaEventRecord(ev[phase].back().second, st));
  }
  void totals(float* h_ms) {
    if (!on) return;
    B200_CUDA(cudaStreamSynchronize(st));
    for (int p = 0; p < 2; ++p) {
      float s = 0.f;
      for (auto& q : ev[p]) { float ms = 0.f; B200_CUDA(cudaEventElapsedTime(&ms, q.first, q.second)); s += ms; }
      h_ms[p] = s;
    }
  }
};

}  // namespace rsvd
}  // namespace b200

using namespace b200;
using namespace b200::rsvd;

extern "C" {

int b200_csr_spmm_dense_device(int64_t n_rows, const int32_t* d_ptr, const int32_t* d_idx, const float* d_val, const float* d_X,
                               int ld, float* d_Y, void* stream) {
  return guarded([&] {
    B200_REQUIRE(n_rows >= 0 && ld >= 4 && ld % 4 == 0 && ld <= MAX_L, "b200_csr_spmm_dense_device: ld must be a multiple of 4 in [4, %d]", MAX_L);
    B200_REQUIRE(n_rows == 0 || (d_ptr && d_X && d_Y), "b200_csr_spmm_dense_device: NULL pointer");
    spmm(n_rows, d_ptr, d_idx, d_val, d_X, ld, d_Y, (cudaStream_t)stream);
  });
}

int b200_csr_transpose_device(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* d_ptr, const int32_t* d_idx,
                              const float* d_val, int32_t* d_t_ptr, int32_t* d_t_idx, float* d_t_val, void* stream) {
  return guarded([&] {
    B200_REQUIRE(n_rows >= 0 && n_cols > 0 && nnz >= 0 && nnz < (1ll << 31) - 1 && n_rows < (1ll << 31) && n_cols < (1ll << 31) - 1,
                 "b200_csr_transpose_device: sizes out of int32 range");
    B200_REQUIRE(d_t_ptr && (nnz == 0 || (d_ptr && d_idx && d_val && d_t_idx && d_t_val)), "b200_csr_transpose_device: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    B200_CUDA(cudaMemsetAsync(d_t_ptr, 0, sizeof(int) * (size_t)(n_cols + 1), st));
    if (nnz == 0) return;
    const size_t n1 = (size_t)nnz;
    DevBuf<int> rows(n1), pos(n1), cols_sorted(n1), perm(n1), cnt((size_t)n_cols);
    B200_CUDA(cudaMemsetAsync(cnt.get(), 0, sizeof(int) * (size_t)n_cols, st));
    int end_bit = 1;
    while ((1ll << end_bit) < n_cols) ++end_bit;
    size_t tb_sort = 0, tb_scan = 0;
    B200_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tb_sort, d_idx, cols_sorted.get(), pos.get(), perm.get(), (int)nnz, 0, end_bit, st));
    B200_CUDA(cub::DeviceScan::InclusiveSum(nullptr, tb_scan, cnt.get(), d_t_ptr + 1, (int)n_cols, st));
    DevBuf<unsigned char> tmp(std::max(tb_sort, tb_scan) + 16);
    entry_rows_kernel<<<div_up(nnz, 256), 256, 0, st>>>(n_rows, nnz, d_ptr, rows.get(), pos.get(), cnt.get(), d_idx);
    B200_CUDA(cudaGetLastError());
    // LSD radix sort is stable: inside a column the entries keep their row order
    B200_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(), tb_sort, d_idx, cols_sorted.get(), pos.get(), perm.get(), (int)nnz, 0, end_bit, st));
    gather_transpose_kernel<<<div_up(nnz, 256), 256, 0, st>>>(nnz, perm.get(), rows.get(), d_val, d_t_idx, d_t_val);
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cub::DeviceScan::InclusiveSum(tmp.get(), tb_scan, cnt.get(), d_t_ptr + 1, (int)n_cols, st));
    count_launch(8);
    B200_CUDA(cudaStreamSynchronize(st));  // the scratch buffers are freed on return
  });
}

int b200_orthonormalize_device(int64_t n, int l, int ld, float* d_Y, uint32_t seed, int32_t* h_breakdowns, void* stream) {
  return guarded([&] {
    B200_REQUIRE(n > 0 && l >= 1 && l <= MAX_L && ld >= l && ld % 4 == 0 && l <= n && d_Y,
                 "b200_orthonormalize_device: need 1 <= l <= min(n, %d), ld >= l a multiple of 4", MAX_L);
    cudaStream_t st = (cudaStream_t)stream;
    DevBuf<float> tmp((size_t)n * ld);
    B200_CUDA(cudaMemsetAsync(tmp.get(), 0, sizeof(float) * tmp.n, st));
    Work w(n, l);
    const int b = orthonormalize(w, n, l, ld, d_Y, tmp.get(), seed, st);
    B200_CUDA(cudaStreamSynchronize(st));
    if (h_breakdowns) *h_breakdowns = b;
  });
}

int b200_rsvd_range_device(int64_t n_rows, int64_t n_cols, const int32_t* d_ptr, const int32_t* d_idx, const float* d_val,
                           const int32_t* d_t_ptr, const int32_t* d_t_idx, const float* d_t_val, const float* d_omega, int l, int ld,
                           int n_iter, uint32_t seed, float* d_Q, float* d_Qb, double* d_Rb, float* h_ms, int32_t* h_breakdowns,
                           void* stream) {
  return guarded([&] {
    B200_REQUIRE(l >= 1 && l <= n_rows && l <= n_cols && ld >= l && ld % 4 == 0 && ld <= MAX_L && n_iter >= 0,
                 "b200_rsvd_range_device: need 1 <= l <= min(n_rows, n_cols), ld >= l a multiple of 4, ld <= %d", MAX_L);
    B200_REQUIRE(d_ptr && d_t_ptr && d_omega && d_Q && d_Qb && d_Rb, "b200_rsvd_range_device: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nb = (size_t)n_rows * ld, mb = (size_t)n_cols * ld;
    DevBuf<float> ntmp(nb), mtmp(mb), bt(mb);
    B200_CUDA(cudaMemsetAsync(ntmp.get(), 0, sizeof(float) * nb, st));
    B200_CUDA(cudaMemsetAsync(mtmp.get(), 0, sizeof(float) * mb, st));
    B200_CUDA(cudaMemsetAsync(d_Q, 0, sizeof(float) * nb, st));
    B200_CUDA(cudaMemcpyAsync(d_Qb, d_omega, sizeof(float) * mb, cudaMemcpyDeviceToDevice, st));
    Work w(n_rows, l);
    Timer tm(h_ms != nullptr, st);
    int breakdowns = 0;
    unsigned pass_seed = seed;
    // sklearn's _randomized_range_finder: n_iter x (A Q, normalise, A^T Q, normalise), then QR(A Q)
    for (int it = 0; it <= n_iter; ++it) {
      tm.begin(0); spmm(n_rows, d_ptr, d_idx, d_val, d_Qb, ld, d_Q, st); tm.end(0);
      tm.begin(1); breakdowns += orthonormalize(w, n_rows, l, ld, d_Q, ntmp.get(), pass_seed++, st); tm.end(1);
      if (it == n_iter) break;
      tm.begin(0); spmm(n_cols, d_t_ptr, d_t_idx, d_t_val, d_Q, ld, d_Qb, st); tm.end(0);
      tm.begin(1); breakdowns += orthonormalize(w, n_cols, l, ld, d_Qb, mtmp.get(), pass_seed++, st); tm.end(1);
    }
    // B^T = A^T Q = Qb Rb with Rb = Qb^T B^T formed explicitly (a refilled column keeps B^T = Qb Rb exact)
    tm.begin(0); spmm(n_cols, d_t_ptr, d_t_idx, d_t_val, d_Q, ld, bt.get(), st); tm.end(0);
    tm.begin(1);
    B200_CUDA(cudaMemcpyAsync(d_Qb, bt.get(), sizeof(float) * mb, cudaMemcpyDeviceToDevice, st));
    breakdowns += orthonormalize(w, n_cols, l, ld, d_Qb, mtmp.get(), pass_seed++, st);
    w.xty(n_cols, d_Qb, bt.get(), ld, st);
    B200_CUDA(cudaMemcpyAsync(d_Rb, w.G.get(), sizeof(double) * l * l, cudaMemcpyDeviceToDevice, st));
    tm.end(1);
    tm.totals(h_ms);
    B200_CUDA(cudaStreamSynchronize(st));
    if (h_breakdowns) *h_breakdowns = breakdowns;
  });
}

int b200_rsvd_finish_device(int64_t n_rows, int64_t n_cols, const float* d_Q, const float* d_Qb, int l, int ld, const double* h_W,
                            const double* h_Z, const float* h_sigma, int k, int transpose, int scale_item_side,
                            float* d_user_factors, float* d_item_factors, void* stream) {
  return guarded([&] {
    B200_REQUIRE(n_rows >= 1 && n_cols >= 1 && l >= 1 && l <= MAX_L && ld >= l && k >= 1 && k <= l,
                 "b200_rsvd_finish_device: need 1 <= k <= l <= %d", MAX_L);
    B200_REQUIRE(d_Q && d_Qb && h_W && h_Z && h_sigma && d_user_factors && d_item_factors, "b200_rsvd_finish_device: NULL pointer");
    cudaStream_t st = (cudaStream_t)stream;
    DevBuf<double> W((size_t)l * l), Z((size_t)l * l);
    DevBuf<float> sigma((size_t)k), sign((size_t)k);
    B200_CUDA(cudaMemcpyAsync(W.get(), h_W, sizeof(double) * l * l, cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(Z.get(), h_Z, sizeof(double) * l * l, cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemcpyAsync(sigma.get(), h_sigma, sizeof(float) * k, cudaMemcpyHostToDevice, st));
    // left factor of A = Q W, right factor = Qb Z (first k columns); A = M^T when transposed
    float* left = transpose ? d_item_factors : d_user_factors;
    float* right = transpose ? d_user_factors : d_item_factors;
    tall_small(n_rows, l, k, d_Q, ld, W.get(), l, left, k, st);
    tall_small(n_cols, l, k, d_Qb, ld, Z.get(), l, right, k, st);
    const long long n_user = transpose ? n_cols : n_rows, n_item = transpose ? n_rows : n_cols;
    const long long chunk = 1024;
    const int parts = (int)div_up(n_user, chunk);
    DevBuf<float> pmax((size_t)parts * k);
    DevBuf<long long> parg((size_t)parts * k);
    colmax_partial_kernel<<<dim3(div_up(k, 128), parts), 128, 0, st>>>(n_user, k, d_user_factors, k, chunk, pmax.get(), parg.get());
    B200_CUDA(cudaGetLastError());
    colsign_kernel<<<div_up(k, 128), 128, 0, st>>>(k, parts, pmax.get(), parg.get(), d_user_factors, k, sign.get());
    B200_CUDA(cudaGetLastError());
    scale_cols_kernel<<<div_up(n_user * k, 256), 256, 0, st>>>(n_user, k, d_user_factors, sign.get(), nullptr);
    B200_CUDA(cudaGetLastError());
    scale_cols_kernel<<<div_up(n_item * k, 256), 256, 0, st>>>(n_item, k, d_item_factors, sign.get(), scale_item_side ? sigma.get() : nullptr);
    B200_CUDA(cudaGetLastError());
    count_launch(4);
    B200_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
