// K2: matrix-factorisation SGD epochs (BPR-MF and FunkSVD), sm_100a.
//
// Replaces MatrixFactorization/Cython/MatrixFactorization_Cython_Epoch.pyx:
//   epochIteration_Cython_BPR_SGD :583-678, epochIteration_Cython_FUNK_SVD_SGD :289-390,
//   _apply_minibatch_updates_to_latent_factors :773-832, adaptive_gradient :838-876,
//   sampleBPR_Cython :943-987, sampleMSE_Cython :881-938.
//
// Two execution modes (DESIGN.md "K2"):
//   * mini-batch (the reference's semantics, exactly): parameters are frozen inside a batch, every sample's
//     gradient is accumulated into per-row accumulators, then every touched row takes one step with the mean
//     gradient (divided by batch_size, pyx:805,828) through the adaptive rule.  One persistent cooperative
//     kernel runs the whole epoch: phase 1 (one warp per sample: three coalesced row gathers, warp-shuffle dot,
//     vector RED.ADD into the accumulators), grid sync, phase 2 (one warp per touched row), grid sync.
//     The sample stream is either replayed on the host with glibc's rand() (bit-compatible with the reference's
//     libc calls) or drawn on the device with Philox4x32-10.
//     Without bias terms the same semantics run as a DATAFLOW (mf_dataflow_kernel, the default): the only true
//     dependences between batches are rows touched again by a later batch (a batch of 1000 touches 3000 of 1.2 M
//     rows at C5), so instead of two grid-wide barriers per batch every (row, batch) pair carries a precomputed
//     expected hit count and the batch that touched the row before; a sample waits until exactly that earlier
//     update is visible, the last sample to hit a row in a batch applies the row's step, and a row hit once in its
//     batch (the common case) is stepped straight from registers without an accumulator round trip.
//   * hogwild: no batch barrier -- every warp applies its sample's update immediately (the reference's
//     batch_size=1 recursion run concurrently; races between warps are the usual Hogwild races).
// Roofline: HBM; bytes per BPR sample = 6 * f * 4 (three rows read, three accumulator rows RMW).
#include <cooperative_groups.h>
#include <cub/device/device_radix_sort.cuh>
#include <stdlib.h>

#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace b200 {
namespace mf {

enum Algo { MF_BPR = 0, FUNK_SVD = 1 };
enum SgdMode { SGD = 0, ADAGRAD = 1, RMSPROP = 2, ADAM = 3 };

struct Params {
  int n_users, n_items, f, batch_size, algorithm, use_bias, sgd_mode, hogwild;
  float lr, user_reg, item_reg, bias_reg, positive_reg, negative_reg;
  float gamma, beta1, beta2;
  double b1_pow, b2_pow;  // adam powers at the start of the epoch
  float *U, *V, *bu, *bi, *mu;
  // batch gradient sums are fp64 like pyx:305-354: a double atomic sum is order-independent to ~1e-16 relative, so the
  // mini-batch mode is run-to-run deterministic at the fp32 precision of the parameters (fp32 RED.ADD was not: the
  // summation order of a row's samples changed the rounded sum, and Adam's m/(sqrt(v)+eps) amplified it)
  double *accU, *accV, *accbu, *accbi, *accmu;
  float *cU, *cV, *cbu, *cbi, *cmu;                                    // adagrad / rmsprop cache
  float *m1U, *m2U, *m1V, *m2V, *m1bu, *m2bu, *m1bi, *m2bi, *m1mu, *m2mu;  // adam
  int *flagI, *flagU, *listI, *listU, *cnt;  // cnt[4]: items/users counters, double-buffered by batch parity
  const int* su; const int* si; const int* sj; const float* sr;  // sample stream of the epoch
  long long n_batches;
  double* pow_out;  // [2] adam powers after the epoch
  // dataflow mode: per row (users first, then items at n_users + i) the batch whose update is in place / arrivals of the
  // current batch; per sample slot (sample * slots + k) the batch that touched the row before and the row's hit count in
  // this batch; per batch the adam bias corrections
  int *applied, *arrived;
  const int *slot_prev, *slot_expect;
  const float *inv1_b, *inv2_b;
};

struct AdaptCtx {
  int mode;
  float gamma, beta1, beta2, inv1, inv2;  // inv = 1 / (1 - beta^t)
};

// pyx:838-876 on one element; c / m1 / m2 point at this element's state
__device__ __forceinline__ float adapt(const AdaptCtx& a, float g, float* c, float* m1, float* m2) {
  if (a.mode == ADAGRAD) {
    const float cc = *c + g * g;
    *c = cc;
    return g / (sqrtf(cc) + 1e-8f);
  } else if (a.mode == RMSPROP) {
    const float cc = *c * a.gamma + (1.f - a.gamma) * g * g;
    *c = cc;
    return g / (sqrtf(cc) + 1e-8f);
  } else if (a.mode == ADAM) {
    const float mm1 = *m1 * a.beta1 + (1.f - a.beta1) * g;
    const float mm2 = *m2 * a.beta2 + (1.f - a.beta2) * g * g;
    *m1 = mm1;
    *m2 = mm2;
    return (mm1 * a.inv1) / (sqrtf(mm2 * a.inv2) + 1e-8f);
  }
  return g;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

__device__ __forceinline__ void red_add4(float* addr, float4 v) {
#if __CUDA_ARCH__ >= 900
  atomicAdd(reinterpret_cast<float4*>(addr), v);
#else
  atomicAdd(addr, v.x); atomicAdd(addr + 1, v.y); atomicAdd(addr + 2, v.z); atomicAdd(addr + 3, v.w);
#endif
}

__device__ __forceinline__ void touch(int* flag, int* list, int* counter, int row) {
  if (atomicExch(flag + row, 1) == 0) list[atomicAdd(counter, 1)] = row;
}

// ---- phase 1: gradients of one sample, accumulated (mini-batch mode)
template <bool VEC4>
__device__ __forceinline__ void bpr_accumulate(const Params& p, int u, int i, int j, int lane) {
  const int f = p.f;
  const float* Uu = p.U + (size_t)u * f;
  const float* Vi = p.V + (size_t)i * f;
  const float* Vj = p.V + (size_t)j * f;
  float x = 0.f;
  if (VEC4) {
    for (int q = lane * 4; q < f; q += 128) {
      const float4 a = *reinterpret_cast<const float4*>(Uu + q), b = *reinterpret_cast<const float4*>(Vi + q),
                   c = *reinterpret_cast<const float4*>(Vj + q);
      x += a.x * (b.x - c.x) + a.y * (b.y - c.y) + a.z * (b.z - c.z) + a.w * (b.w - c.w);
    }
  } else {
    for (int q = lane; q < f; q += 32) x += Uu[q] * (Vi[q] - Vj[q]);
  }
  x = warp_sum(x);
  const float sig = 1.f / (1.f + expf(x));  // pyx:622
  double* aU = p.accU + (size_t)u * f;
  double* aI = p.accV + (size_t)i * f;
  double* aJ = p.accV + (size_t)j * f;
  const double sg = (double)sig, rp = (double)p.positive_reg, rn = (double)p.negative_reg, ru = (double)p.user_reg;
  for (int q = lane; q < f; q += 32) {  // consecutive lanes -> consecutive 8-byte RED.ADD.F64 (coalesced)
    const double a = (double)Uu[q], b = (double)Vi[q], c = (double)Vj[q];
    atomicAdd(aI + q, sg * a - rp * b);        // pyx:633
    atomicAdd(aJ + q, -sg * a - rn * c);       // pyx:634
    atomicAdd(aU + q, sg * (b - c) - ru * a);  // pyx:635
  }
}

template <bool VEC4>
__device__ __forceinline__ void mse_accumulate(const Params& p, int u, int i, float r, int lane) {
  const int f = p.f;
  const float* Uu = p.U + (size_t)u * f;
  const float* Vi = p.V + (size_t)i * f;
  float x = 0.f;
  if (VEC4) {
    for (int q = lane * 4; q < f; q += 128) {
      const float4 a = *reinterpret_cast<const float4*>(Uu + q), b = *reinterpret_cast<const float4*>(Vi + q);
      x += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
    }
  } else {
    for (int q = lane; q < f; q += 32) x += Uu[q] * Vi[q];
  }
  x = warp_sum(x);
  if (p.use_bias) x += p.mu[0] + p.bu[u] + p.bi[i];  // pyx:313-316
  const float err = r - x;
  const double er = (double)err;
  if (p.use_bias && lane == 0) {  // pyx:332-339
    const double rb = (double)p.bias_reg;
    atomicAdd(p.accmu, er - rb * (double)p.mu[0]);
    atomicAdd(p.accbi + i, er - rb * (double)p.bi[i]);
    atomicAdd(p.accbu + u, er - rb * (double)p.bu[u]);
  }
  double* aU = p.accU + (size_t)u * f;
  double* aI = p.accV + (size_t)i * f;
  const double rp = (double)p.positive_reg, ru = (double)p.user_reg;
  for (int q = lane; q < f; q += 32) {
    const double a = (double)Uu[q], b = (double)Vi[q];
    atomicAdd(aI + q, er * a - rp * b);  // item regulariser is positive_reg, not item_reg (pyx:349)
    atomicAdd(aU + q, er * b - ru * a);
  }
}

// ---- phase 2: one touched row takes its step (pyx:792-832)
__device__ __forceinline__ void apply_row(const Params& p, const AdaptCtx& ad, float* P, double* acc, float* c, float* m1,
                                          float* m2, size_t row, int lane, double inv_bs) {
  const int f = p.f;
  const size_t o = row * (size_t)f;
  for (int q = lane; q < f; q += 32) {
    float g = (float)(acc[o + q] * inv_bs);
    g = adapt(ad, g, c ? c + o + q : nullptr, m1 ? m1 + o + q : nullptr, m2 ? m2 + o + q : nullptr);
    P[o + q] += p.lr * g;
    acc[o + q] = 0.0;
  }
}

__device__ __forceinline__ void apply_scalar(const Params& p, const AdaptCtx& ad, float* P, double* acc, float* c, float* m1,
                                             float* m2, size_t k, double inv_bs) {
  float g = (float)(acc[k] * inv_bs);
  g = adapt(ad, g, c ? c + k : nullptr, m1 ? m1 + k : nullptr, m2 ? m2 + k : nullptr);
  P[k] += p.lr * g;
  acc[k] = 0.0;
}

template <bool VEC4>
__global__ void __launch_bounds__(256) mf_epoch_kernel(const Params p) {
  cg::grid_group grid = cg::this_grid();
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const double inv_bs = 1.0 / (double)p.batch_size;
  double b1p = p.b1_pow, b2p = p.b2_pow;
  AdaptCtx ad;
  ad.mode = p.sgd_mode; ad.gamma = p.gamma; ad.beta1 = p.beta1; ad.beta2 = p.beta2;
  for (long long b = 0; b < p.n_batches; ++b) {
    int* cnt = p.cnt + 2 * (int)(b & 1);
    // ---------------- phase 1
    for (long long s = warp; s < p.batch_size; s += n_warps) {
      const long long g = b * p.batch_size + s;
      const int u = p.su[g], i = p.si[g];
      if (p.algorithm == MF_BPR) {
        const int j = p.sj[g];
        if (lane == 0) { touch(p.flagI, p.listI, cnt, i); touch(p.flagI, p.listI, cnt, j); touch(p.flagU, p.listU, cnt + 1, u); }
        bpr_accumulate<VEC4>(p, u, i, j, lane);
      } else {
        if (lane == 0) { touch(p.flagI, p.listI, cnt, i); touch(p.flagU, p.listU, cnt + 1, u); }
        mse_accumulate<VEC4>(p, u, i, p.sr[g], lane);
      }
    }
    grid.sync();
    // ---------------- phase 2
    ad.inv1 = (float)(1.0 / (1.0 - b1p));
    ad.inv2 = (float)(1.0 / (1.0 - b2p));
    const int nI = cnt[0], nU = cnt[1];
    if (p.use_bias && warp == 0 && lane == 0) apply_scalar(p, ad, p.mu, p.accmu, p.cmu, p.m1mu, p.m2mu, 0, inv_bs);
    for (long long t = warp; t < nI + nU; t += n_warps) {
      if (t < nI) {
        const int k = p.listI[t];
        if (p.use_bias && lane == 0) apply_scalar(p, ad, p.bi, p.accbi, p.cbi, p.m1bi, p.m2bi, k, inv_bs);
        apply_row(p, ad, p.V, p.accV, p.cV, p.m1V, p.m2V, k, lane, inv_bs);
        if (lane == 0) p.flagI[k] = 0;
      } else {
        const int k = p.listU[t - nI];
        if (p.use_bias && lane == 0) apply_scalar(p, ad, p.bu, p.accbu, p.cbu, p.m1bu, p.m2bu, k, inv_bs);
        apply_row(p, ad, p.U, p.accU, p.cU, p.m1U, p.m2U, k, lane, inv_bs);
        if (lane == 0) p.flagU[k] = 0;
      }
    }
    if (warp == 0 && lane == 0) { int* nxt = p.cnt + 2 * (int)((b + 1) & 1); nxt[0] = 0; nxt[1] = 0; }
    if (p.sgd_mode == ADAM) { b1p *= (double)p.beta1; b2p *= (double)p.beta2; }  // once per batch, pyx:649-652
    grid.sync();
  }
  if (warp == 0 && lane == 0) { p.pow_out[0] = b1p; p.pow_out[1] = b2p; p.cnt[0] = p.cnt[1] = p.cnt[2] = p.cnt[3] = 0; }
}

// ---- hogwild: every warp applies its samples' updates at once (batch_size = 1 recursion, concurrent)
__global__ void __launch_bounds__(256) mf_hogwild_kernel(const Params p, long long n_samples) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int f = p.f;
  AdaptCtx ad;
  ad.mode = p.sgd_mode; ad.gamma = p.gamma; ad.beta1 = p.beta1; ad.beta2 = p.beta2;
  for (long long g = warp; g < n_samples; g += n_warps) {
    if (p.sgd_mode == ADAM) {  // the reference advances the powers once per (size-1) batch
      ad.inv1 = (float)(1.0 / (1.0 - p.b1_pow * pow((double)p.beta1, (double)g)));
      ad.inv2 = (float)(1.0 / (1.0 - p.b2_pow * pow((double)p.beta2, (double)g)));
    }
    const int u = p.su[g], i = p.si[g];
    float* Uu = p.U + (size_t)u * f;
    float* Vi = p.V + (size_t)i * f;
    if (p.algorithm == MF_BPR && p.sgd_mode == SGD && (f & 3) == 0) {
      // plain-SGD BPR, rows as float4: one 16-byte load and store per lane and row for f = 128
      const int j = p.sj[g];
      float* Vj = p.V + (size_t)j * f;
      float x = 0.f;
      for (int q = lane * 4; q < f; q += 128) {
        const float4 a = *reinterpret_cast<const float4*>(Uu + q), b = *reinterpret_cast<const float4*>(Vi + q),
                     c = *reinterpret_cast<const float4*>(Vj + q);
        x += a.x * (b.x - c.x) + a.y * (b.y - c.y) + a.z * (b.z - c.z) + a.w * (b.w - c.w);
      }
      x = warp_sum(x);
      const float sig = 1.f / (1.f + expf(x));
      const float lr = p.lr;
      for (int q = lane * 4; q < f; q += 128) {
        const float4 a = *reinterpret_cast<const float4*>(Uu + q), b = *reinterpret_cast<const float4*>(Vi + q),
                     c = *reinterpret_cast<const float4*>(Vj + q);
        // deltas go through RED.ADD so that concurrent samples sharing a row add up instead of overwriting each other
        red_add4(Vi + q, make_float4(lr * (sig * a.x - p.positive_reg * b.x), lr * (sig * a.y - p.positive_reg * b.y),
                                     lr * (sig * a.z - p.positive_reg * b.z), lr * (sig * a.w - p.positive_reg * b.w)));
        red_add4(Vj + q, make_float4(lr * (-sig * a.x - p.negative_reg * c.x), lr * (-sig * a.y - p.negative_reg * c.y),
                                     lr * (-sig * a.z - p.negative_reg * c.z), lr * (-sig * a.w - p.negative_reg * c.w)));
        red_add4(Uu + q, make_float4(lr * (sig * (b.x - c.x) - p.user_reg * a.x), lr * (sig * (b.y - c.y) - p.user_reg * a.y),
                                     lr * (sig * (b.z - c.z) - p.user_reg * a.z), lr * (sig * (b.w - c.w) - p.user_reg * a.w)));
      }
    } else if (p.algorithm == MF_BPR) {
      const int j = p.sj[g];
      float* Vj = p.V + (size_t)j * f;
      float x = 0.f;
      for (int q = lane; q < f; q += 32) x += Uu[q] * (Vi[q] - Vj[q]);
      x = warp_sum(x);
      const float sig = 1.f / (1.f + expf(x));
      for (int q = lane; q < f; q += 32) {
        const float a = Uu[q], b = Vi[q], c = Vj[q];
        const size_t oi = (size_t)i * f + q, oj = (size_t)j * f + q, ou = (size_t)u * f + q;
        // items first, then the user, as pyx:792-832 orders the apply
        atomicAdd(Vi + q, p.lr * adapt(ad, sig * a - p.positive_reg * b, p.cV ? p.cV + oi : nullptr, p.m1V ? p.m1V + oi : nullptr, p.m2V ? p.m2V + oi : nullptr));
        atomicAdd(Vj + q, p.lr * adapt(ad, -sig * a - p.negative_reg * c, p.cV ? p.cV + oj : nullptr, p.m1V ? p.m1V + oj : nullptr, p.m2V ? p.m2V + oj : nullptr));
        atomicAdd(Uu + q, p.lr * adapt(ad, sig * (b - c) - p.user_reg * a, p.cU ? p.cU + ou : nullptr, p.m1U ? p.m1U + ou : nullptr, p.m2U ? p.m2U + ou : nullptr));
      }
    } else {
      float x = 0.f;
      for (int q = lane; q < f; q += 32) x += Uu[q] * Vi[q];
      x = warp_sum(x);
      if (p.use_bias) x += p.mu[0] + p.bu[u] + p.bi[i];
      const float err = p.sr[g] - x;
      if (p.use_bias && lane == 0) {
        p.mu[0] += p.lr * adapt(ad, err - p.bias_reg * p.mu[0], p.cmu, p.m1mu, p.m2mu);
        p.bi[i] += p.lr * adapt(ad, err - p.bias_reg * p.bi[i], p.cbi ? p.cbi + i : nullptr, p.m1bi ? p.m1bi + i : nullptr, p.m2bi ? p.m2bi + i : nullptr);
        p.bu[u] += p.lr * adapt(ad, err - p.bias_reg * p.bu[u], p.cbu ? p.cbu + u : nullptr, p.m1bu ? p.m1bu + u : nullptr, p.m2bu ? p.m2bu + u : nullptr);
      }
      for (int q = lane; q < f; q += 32) {
        const float a = Uu[q], b = Vi[q];
        const size_t oi = (size_t)i * f + q, ou = (size_t)u * f + q;
        atomicAdd(Vi + q, p.lr * adapt(ad, err * a - p.positive_reg * b, p.cV ? p.cV + oi : nullptr, p.m1V ? p.m1V + oi : nullptr, p.m2V ? p.m2V + oi : nullptr));
        atomicAdd(Uu + q, p.lr * adapt(ad, err * b - p.user_reg * a, p.cU ? p.cU + ou : nullptr, p.m1U ? p.m1U + ou : nullptr, p.m2U ? p.m2U + ou : nullptr));
      }
    }
  }
}


// =====================================================================================================================
// Dataflow mini-batch mode (same arithmetic and semantics as mf_epoch_kernel, no grid-wide barrier).
//   row ids: user u -> u, item i -> n_users + i.  slot k of sample g: 0 = user, 1 = item i, 2 = item j (BPR).
//   slot_prev[g*S+k]   = the latest batch < batch(g) of this epoch that touches the row, or -1
//   slot_expect[g*S+k] = how many samples of batch(g) touch the row
//   applied[row]       = batch whose step is in place (-1 at epoch start); published with st.release after the row is
//                        written, read with ld.acquire before the row is read; rows and optimiser state move with
//                        .cg accesses (L2 only), so no stale L1 line can be observed
// Progress: warps take samples in increasing order and wait only for steps of earlier batches, each of which is taken by
// one of that batch's samples; with every warp resident (cooperative launch) the smallest unfinished sample never waits.
__device__ __forceinline__ int ld_relaxed(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(int* p, int v) { asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// Ordering: a sample spins on its rows' `applied` words with relaxed loads and then executes ONE fence (acquire side) before
// it reads the rows; after its last write it executes ONE fence (release side) and then publishes with relaxed stores /
// the arrival atomics.  fence + relaxed access is the PTX release / acquire pattern; one fence serves all three rows.

// pyx:838-876 on one element with L2-only accesses to the state
__device__ __forceinline__ float adapt_cg(const AdaptCtx& a, float g, float* c, float* m1, float* m2) {
  if (a.mode == ADAGRAD) {
    const float cc = __ldcg(c) + g * g;
    __stcg(c, cc);
    return g / (sqrtf(cc) + 1e-8f);
  } else if (a.mode == RMSPROP) {
    const float cc = __ldcg(c) * a.gamma + (1.f - a.gamma) * g * g;
    __stcg(c, cc);
    return g / (sqrtf(cc) + 1e-8f);
  } else if (a.mode == ADAM) {
    const float mm1 = __ldcg(m1) * a.beta1 + (1.f - a.beta1) * g;
    const float mm2 = __ldcg(m2) * a.beta2 + (1.f - a.beta2) * g * g;
    __stcg(m1, mm1);
    __stcg(m2, mm2);
    return (mm1 * a.inv1) / (sqrtf(mm2 * a.inv2) + 1e-8f);
  }
  return g;
}

// one row's share of a sample: either the row's whole step (it is hit once in this batch) or a contribution to its sum
struct SlotCtx {
  float* P; double* acc; float *c, *m1, *m2;  // row base pointers (state pointers may be null)
  bool direct;
};
// returns the element's new value when the slot steps directly (the caller stores it), `old` otherwise
__device__ __forceinline__ float slot_element(const Params& p, const AdaptCtx& ad, const SlotCtx& s, int q, float old, double term,
                                              double inv_bs) {
  if (s.direct) {
    float g = (float)(term * inv_bs);  // what apply_row computes from a one-term sum
    g = adapt_cg(ad, g, s.c ? s.c + q : nullptr, s.m1 ? s.m1 + q : nullptr, s.m2 ? s.m2 + q : nullptr);
    return old + p.lr * g;
  }
  atomicAdd(s.acc + q, term);
  return old;
}
// the step of a row whose sum is complete (pyx:792-832), L2-only accesses
__device__ __forceinline__ void apply_row_cg(const Params& p, const AdaptCtx& ad, const SlotCtx& s, int lane, double inv_bs) {
  for (int q = lane; q < p.f; q += 32) {
    float g = (float)(__ldcg(s.acc + q) * inv_bs);
    g = adapt_cg(ad, g, s.c ? s.c + q : nullptr, s.m1 ? s.m1 + q : nullptr, s.m2 ? s.m2 + q : nullptr);
    __stcg(s.P + q, __ldcg(s.P + q) + p.lr * g);
    __stcg(s.acc + q, 0.0);
  }
}
// after the release fence: publish a directly stepped row, or count the arrival at a shared row and, as the last sample
// to arrive, take the row's step
__device__ __forceinline__ void slot_publish(const Params& p, const AdaptCtx& ad, const SlotCtx& s, int row, int expect, int batch,
                                             int lane, double inv_bs) {
  if (s.direct) {
    if (lane == 0) st_relaxed(p.applied + row, batch);
    return;
  }
  int last = 0;
  if (lane == 0) last = (atomicAdd(p.arrived + row, 1) + 1 == expect) ? 1 : 0;
  last = __shfl_sync(0xffffffffu, last, 0);
  if (!last) return;
  __threadfence();  // acquire side of the arrival counter: every contribution to the sum is visible
  apply_row_cg(p, ad, s, lane, inv_bs);
  __threadfence();
  __syncwarp();
  if (lane == 0) {
    p.arrived[row] = 0;
    __threadfence();
    st_relaxed(p.applied + row, batch);
  }
}

// ONE4: n_factors is a multiple of 4 and at most 128 -- every lane owns one float4 of each row, read once
template <bool BPR, bool ONE4>
__global__ void __launch_bounds__(256, 3) mf_dataflow_kernel(const Params p, long long n_samples) {
  constexpr int S = BPR ? 3 : 2;
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int f = p.f, nU = p.n_users;
  const double inv_bs = 1.0 / (double)p.batch_size;
  AdaptCtx ad;
  ad.mode = p.sgd_mode; ad.gamma = p.gamma; ad.beta1 = p.beta1; ad.beta2 = p.beta2; ad.inv1 = ad.inv2 = 1.f;
  const double rp = (double)p.positive_reg, rn = (double)p.negative_reg, rgu = (double)p.user_reg;
  for (long long g = warp; g < n_samples; g += n_warps) {
    const int batch = (int)(g / p.batch_size);
    const int u = p.su[g], i = p.si[g], j = BPR ? p.sj[g] : 0;
    const int ru = u, ri = nU + i, rj = nU + j;
    const long long s0 = g * S;
    const int pu = p.slot_prev[s0], pi = p.slot_prev[s0 + 1], pj = BPR ? p.slot_prev[s0 + 2] : 0;
    const int eu = p.slot_expect[s0], ei = p.slot_expect[s0 + 1], ej = BPR ? p.slot_expect[s0 + 2] : 0;
    if (p.sgd_mode == ADAM) { ad.inv1 = p.inv1_b[batch]; ad.inv2 = p.inv2_b[batch]; }
    // ---- wait for the three rows' previous steps
    {
      unsigned ns = 20;
      for (;;) {
        const int vu = ld_relaxed(p.applied + ru), vi = ld_relaxed(p.applied + ri), vj = BPR ? ld_relaxed(p.applied + rj) : pj;
        if (vu == pu && vi == pi && vj == pj) break;
        __nanosleep(ns);
        if (ns < 640) ns <<= 1;
      }
      __threadfence();
    }
    float* Uu = p.U + (size_t)u * f;
    float* Vi = p.V + (size_t)i * f;
    float* Vj = p.V + (size_t)j * f;
    const size_t ou = (size_t)u * f, oi = (size_t)i * f, oj = (size_t)j * f;
    SlotCtx su_{Uu, p.accU + ou, p.cU ? p.cU + ou : nullptr, p.m1U ? p.m1U + ou : nullptr, p.m2U ? p.m2U + ou : nullptr, eu == 1};
    SlotCtx si_{Vi, p.accV + oi, p.cV ? p.cV + oi : nullptr, p.m1V ? p.m1V + oi : nullptr, p.m2V ? p.m2V + oi : nullptr, ei == 1};
    SlotCtx sj_{Vj, p.accV + oj, p.cV ? p.cV + oj : nullptr, p.m1V ? p.m1V + oj : nullptr, p.m2V ? p.m2V + oj : nullptr, ej == 1};
    if (ONE4) {
      const int q = lane * 4;
      const bool on = q < f;
      float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f), b4 = a4, c4 = a4;
      if (on) {
        a4 = __ldcg(reinterpret_cast<const float4*>(Uu + q));
        b4 = __ldcg(reinterpret_cast<const float4*>(Vi + q));
        if (BPR) c4 = __ldcg(reinterpret_cast<const float4*>(Vj + q));
      }
      float x = BPR ? a4.x * (b4.x - c4.x) + a4.y * (b4.y - c4.y) + a4.z * (b4.z - c4.z) + a4.w * (b4.w - c4.w)
                    : a4.x * b4.x + a4.y * b4.y + a4.z * b4.z + a4.w * b4.w;
      x = warp_sum(x);
      // BPR: sigma = 1 / (1 + e^x), pyx:622; FunkSVD (no bias here): err = r - x, pyx:318
      const double coef = BPR ? (double)(1.f / (1.f + expf(x))) : (double)(p.sr[g] - x);
      if (on) {
        const float af[4] = {a4.x, a4.y, a4.z, a4.w}, bf[4] = {b4.x, b4.y, b4.z, b4.w}, cf[4] = {c4.x, c4.y, c4.z, c4.w};
        float na[4], nb[4], nc[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const double a = (double)af[e], b = (double)bf[e], c = (double)cf[e];
          if (BPR) {
            nb[e] = slot_element(p, ad, si_, q + e, bf[e], coef * a - rp * b, inv_bs);         // pyx:633
            nc[e] = slot_element(p, ad, sj_, q + e, cf[e], -coef * a - rn * c, inv_bs);        // pyx:634
            na[e] = slot_element(p, ad, su_, q + e, af[e], coef * (b - c) - rgu * a, inv_bs);  // pyx:635
          } else {
            nb[e] = slot_element(p, ad, si_, q + e, bf[e], coef * a - rp * b, inv_bs);   // pyx:349 (positive_reg, not item_reg)
            na[e] = slot_element(p, ad, su_, q + e, af[e], coef * b - rgu * a, inv_bs);  // pyx:350
            nc[e] = 0.f;
          }
        }
        if (si_.direct) __stcg(reinterpret_cast<float4*>(Vi + q), make_float4(nb[0], nb[1], nb[2], nb[3]));
        if (BPR && sj_.direct) __stcg(reinterpret_cast<float4*>(Vj + q), make_float4(nc[0], nc[1], nc[2], nc[3]));
        if (su_.direct) __stcg(reinterpret_cast<float4*>(Uu + q), make_float4(na[0], na[1], na[2], na[3]));
      }
    } else {
      float x = 0.f;
      for (int q = lane; q < f; q += 32) x += BPR ? __ldcg(Uu + q) * (__ldcg(Vi + q) - __ldcg(Vj + q)) : __ldcg(Uu + q) * __ldcg(Vi + q);
      x = warp_sum(x);
      const double coef = BPR ? (double)(1.f / (1.f + expf(x))) : (double)(p.sr[g] - x);
      // every element: the terms from the OLD values, then each row's own action
      for (int q = lane; q < f; q += 32) {
        const float af = __ldcg(Uu + q), bf = __ldcg(Vi + q), cf = BPR ? __ldcg(Vj + q) : 0.f;
        const double a = (double)af, b = (double)bf, c = (double)cf;
        if (BPR) {
          const float nb = slot_element(p, ad, si_, q, bf, coef * a - rp * b, inv_bs);
          const float nc = slot_element(p, ad, sj_, q, cf, -coef * a - rn * c, inv_bs);
          const float na = slot_element(p, ad, su_, q, af, coef * (b - c) - rgu * a, inv_bs);
          if (si_.direct) __stcg(Vi + q, nb);
          if (sj_.direct) __stcg(Vj + q, nc);
          if (su_.direct) __stcg(Uu + q, na);
        } else {
          const float nb = slot_element(p, ad, si_, q, bf, coef * a - rp * b, inv_bs);
          const float na = slot_element(p, ad, su_, q, af, coef * b - rgu * a, inv_bs);
          if (si_.direct) __stcg(Vi + q, nb);
          if (su_.direct) __stcg(Uu + q, na);
        }
      }
    }
    // ---- one release fence for all rows, then publish / arrive
    __threadfence();
    __syncwarp();
    slot_publish(p, ad, si_, ri, ei, batch, lane, inv_bs);
    if (BPR) slot_publish(p, ad, sj_, rj, ej, batch, lane, inv_bs);
    slot_publish(p, ad, su_, ru, eu, batch, lane, inv_bs);
  }
}

// ---- multi-GPU exchange of a replicated factor table (dist.ShardedBPR): two fused element-wise passes
// snapshot: d = V - B (this rank's own movement since the last snapshot), D = d (the all-reduce runs in place on D),
// B = V.  The training kernel may be writing V concurrently (Hogwild): whatever this pass reads is what B records, so
// d + B_old == B_new exactly and later writes land in the next delta.
__global__ void mf_delta_snapshot_kernel(const float4* __restrict__ V, float4* __restrict__ B, float4* __restrict__ d,
                                         float4* __restrict__ D, long long n4) {
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += (long long)gridDim.x * blockDim.x) {
    const float4 v = __ldcg(V + k), b = B[k];
    const float4 x = make_float4(v.x - b.x, v.y - b.y, v.z - b.z, v.w - b.w);
    d[k] = x;
    D[k] = x;
    B[k] = v;
  }
}
// apply: t = D - d (the other ranks' movement); V += t with RED.ADD (the training kernel keeps updating V), B += t
__global__ void mf_delta_apply_kernel(float4* __restrict__ V, float4* __restrict__ B, const float4* __restrict__ D,
                                      const float4* __restrict__ d, long long n4) {
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += (long long)gridDim.x * blockDim.x) {
    const float4 a = D[k], o = d[k];
    const float4 t = make_float4(a.x - o.x, a.y - o.y, a.z - o.z, a.w - o.w);
    red_add4(reinterpret_cast<float*>(V + k), t);
    float4 b = B[k];
    b.x += t.x; b.y += t.y; b.z += t.z; b.w += t.w;
    B[k] = b;
  }
}

// keys of the (row, batch) pairs of an epoch's sample stream: row << bbits | batch; value = slot id
template <bool BPR>
__global__ void mf_slot_keys_kernel(const int* __restrict__ su, const int* __restrict__ si, const int* __restrict__ sj, long long n,
                                    int n_users, int batch_size, int bbits, unsigned long long* keys, int* vals) {
  constexpr int S = BPR ? 3 : 2;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n) return;
  const unsigned long long b = (unsigned long long)(g / batch_size);
  keys[g * S] = ((unsigned long long)su[g] << bbits) | b;
  keys[g * S + 1] = ((unsigned long long)(n_users + si[g]) << bbits) | b;
  if (BPR) keys[g * S + 2] = ((unsigned long long)(n_users + sj[g]) << bbits) | b;
  for (int k = 0; k < S; ++k) vals[g * S + k] = (int)(g * S + k);
}

// sorted keys -> per slot: previous batch of the row, hit count of the (row, batch) run.  The head of a run walks it.
__global__ void mf_deps_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ vals, long long m, int bbits,
                               int* slot_prev, int* slot_expect) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  const unsigned long long key = keys[t];
  if (t > 0 && keys[t - 1] == key) return;
  int prev = -1;
  if (t > 0 && (keys[t - 1] >> bbits) == (key >> bbits)) prev = (int)(keys[t - 1] & ((1ull << bbits) - 1ull));
  long long e = t + 1;
  while (e < m && keys[e] == key) ++e;
  const int cnt = (int)(e - t);
  for (long long k = t; k < e; ++k) {
    const int slot = vals[k];
    slot_prev[slot] = prev;
    slot_expect[slot] = cnt;
  }
}

// ---- device sampler: Philox4x32-10 (common.cuh), counter = (sample index, draw block), key = (seed, epoch)

struct Draws {
  unsigned long long idx; unsigned seed, epoch, blk; uint4 cur; int pos;
  __device__ Draws(unsigned long long i, unsigned s, unsigned e) : idx(i), seed(s), epoch(e), blk(0), pos(4) {}
  __device__ unsigned next() {
    if (pos == 4) { cur = philox(idx, blk++, seed, epoch); pos = 0; }
    const unsigned v = pos == 0 ? cur.x : (pos == 1 ? cur.y : (pos == 2 ? cur.z : cur.w));
    ++pos;
    return v;
  }
};

// same acceptance rules as sampleBPR_Cython / sampleMSE_Cython (users with 0 < profile < n_items; negative item
// not in the sorted profile, binary search instead of the linear scan), different random stream
__global__ void mf_sample_kernel(const int* __restrict__ indptr, const int* __restrict__ indices, const float* __restrict__ data,
                                 int user_lo, int n_users, int n_items, int algorithm, float quota, long long n_samples, unsigned seed,
                                 unsigned epoch, int* su, int* si, int* sj, float* sr) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_samples) return;
  Draws d((unsigned long long)g, seed, epoch);
  int u, s, n;
  do {
    u = user_lo + (int)(d.next() % (unsigned)n_users);  // n_users = size of this rank's user shard
    s = indptr[u];
    n = indptr[u + 1] - s;
  } while (n == 0 || n == n_items);
  bool positive = true;
  if (algorithm == FUNK_SVD && quota != 0.f) positive = (float)(d.next() >> 8) * (1.f / 16777216.f) <= quota;
  int item;
  float r = 0.f;
  if (algorithm == MF_BPR || positive) {
    const int k = (int)(d.next() % (unsigned)n);
    item = indices[s + k];
    if (algorithm == FUNK_SVD) r = data[s + k];
  }
  if (algorithm == MF_BPR || !positive) {
    int neg;
    while (true) {
      neg = (int)(d.next() % (unsigned)n_items);
      int lo = 0, hi = n;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (indices[s + mid] < neg) lo = mid + 1; else hi = mid; }
      if (lo == n || indices[s + lo] != neg) break;
    }
    if (algorithm == MF_BPR) sj[g] = neg; else { item = neg; r = 0.f; }
  }
  su[g] = u;
  si[g] = item;
  if (algorithm == FUNK_SVD) sr[g] = r;
}


// =====================================================================================================================
// glibc stream on the device.  The reference draws its samples with libc rand() (sampleBPR_Cython pyx:943-987,
// sampleMSE_Cython :881-938): a sequential recurrence feeding rejection loops, so sample g's first draw depends on how many
// draws every earlier sample consumed.  The raw stream itself is cheap to produce in order (1 ns per draw on the host);
// what made the host replay slow (160 ms per C5 epoch) are the dependent memory lookups of the acceptance rules.  Here:
//   1. the host appends raw draws to a pinned buffer and uploads them;
//   2. glibc_len_kernel: for EVERY position p of the buffer, how many draws a sample STARTING at p would consume;
//   3. pointer doubling: J_0[p] = p + len[p], J_{k+1} = J_k o J_k, so that any number of samples can be skipped at once;
//   4. glibc_emit_kernel: sample g starts where the binary expansion of g leads from position 0; it is re-evaluated there
//      and written out.  The number of draws the epoch consumed tells the host where the next epoch's stream begins.
// Bit-identical to the host replay (same draws, same rules); tests compare the two.
struct GlibcView {
  const int* __restrict__ raw; int R;  // draws raw[0 .. R)
  const int* __restrict__ indptr; const int* __restrict__ indices; const float* __restrict__ data;
  int n_users, n_items, algorithm; float quota;
};

// the sample starting at raw position p: returns the position after its last draw (> R when the buffer ran out)
__device__ __forceinline__ int glibc_sample_at(const GlibcView& v, int p, int* u_out, int* i_out, int* j_out, float* r_out) {
  int q = p;
  int u = 0, s = 0, n = 0;
  for (;;) {  // pyx:952-960 / :890-898: users with an empty or a full profile are redrawn
    if (q >= v.R) return v.R + 1;
    u = v.raw[q++] % v.n_users;
    s = v.indptr[u];
    n = v.indptr[u + 1] - s;
    if (n != 0 && n != v.n_items) break;
  }
  bool positive = true;
  if (v.algorithm == FUNK_SVD && v.quota != 0.f) {  // pyx:901
    if (q >= v.R) return v.R + 1;
    positive = (double)v.raw[q++] <= (double)v.quota * 2147483647.0;
  }
  int item = -1;
  float r = 0.f;
  if (v.algorithm == MF_BPR || positive) {
    if (q >= v.R) return v.R + 1;
    const int k = v.raw[q++] % n;
    item = v.indices[s + k];
    if (v.algorithm == FUNK_SVD) r = v.data[s + k];
  }
  if (v.algorithm == MF_BPR || !positive) {
    int neg;
    for (;;) {
      if (q >= v.R) return v.R + 1;
      neg = v.raw[q++] % v.n_items;
      int lo = 0, hi = n;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (v.indices[s + mid] < neg) lo = mid + 1; else hi = mid; }
      if (lo == n || v.indices[s + lo] != neg) break;
    }
    if (v.algorithm == MF_BPR) { if (j_out) *j_out = neg; } else { item = neg; r = 0.f; }
  }
  if (u_out) *u_out = u;
  if (i_out) *i_out = item;
  if (r_out) *r_out = r;
  return q;
}

__global__ void glibc_len_kernel(const GlibcView v, int* __restrict__ nxt) {  // nxt[p] = start of the following sample; nxt[R] = R
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p > v.R) return;
  nxt[p] = p == v.R ? v.R : min(glibc_sample_at(v, p, nullptr, nullptr, nullptr, nullptr), v.R);
}

__global__ void glibc_double_kernel(const int* __restrict__ jk, int R, int* __restrict__ jk1) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p <= R) jk1[p] = jk[jk[p]];
}

// sample g: follow the binary expansion of g through the jump tables (tables[k] = J_k, (R + 1) ints each), evaluate, store
__global__ void glibc_emit_kernel(const GlibcView v, const int* __restrict__ tables, int levels, long long n_samples, int* su, int* si,
                                  int* sj, float* sr, int* consumed) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_samples) return;
  int p = 0;
  for (int k = 0; k < levels; ++k)
    if ((g >> k) & 1) p = tables[(size_t)k * (v.R + 1) + p];
  int u = 0, i = 0, j = 0;
  float r = 0.f;
  const int q = p < v.R ? glibc_sample_at(v, p, &u, &i, &j, &r) : v.R + 1;
  su[g] = u; si[g] = i;
  if (v.algorithm == MF_BPR) sj[g] = j; else sr[g] = r;
  if (q > v.R) atomicMax(consumed, 0x7FFFFFFF);  // the buffer ran out somewhere: the host extends it and repeats
  else if (g == n_samples - 1) atomicMax(consumed, q);
}

// host replay of glibc srand()/rand() (TYPE_3 additive feedback, r[i] = r[i-31] + r[i-3], 310 discarded, >> 1)
struct GlibcRand {
  int32_t r[31];
  int f = 3, b = 0;
  void seed(unsigned s) {
    int32_t word = s == 0 ? 1 : (int32_t)s;
    r[0] = word;
    for (int i = 1; i < 31; ++i) {
      const long hi = word / 127773, lo = word % 127773;
      long w = 16807 * lo - 2836 * hi;
      if (w < 0) w += 2147483647;
      word = (int32_t)w;
      r[i] = word;
    }
    f = 3; b = 0;
    for (int i = 0; i < 310; ++i) next_raw();
  }
  uint32_t next_raw() {
    const uint32_t v = (uint32_t)r[f] + (uint32_t)r[b];
    r[f] = (int32_t)v;
    if (++f == 31) f = 0;
    if (++b == 31) b = 0;
    return v;
  }
  int next() { return (int)(next_raw() >> 1); }
};

}  // namespace mf
}  // namespace b200

using namespace b200;
using namespace b200::mf;

struct b200_mf_s {
  Params p{};
  int sampler = 0;  // 0 glibc replay on the host, 1 Philox on the device
  unsigned seed = 1;
  unsigned epoch = 0;
  long long nnz = 0;
  float quota = 0.5f;
  GlibcRand rng;
  std::vector<int> h_indptr, h_indices;
  std::vector<float> h_data;
  DevBuf<int> d_indptr, d_indices;
  DevBuf<float> d_data;
  std::vector<DevBuf<float>> fbufs;  // owns every float device array referenced by p
  std::vector<DevBuf<double>> dbufs;  // the fp64 gradient accumulators of the mini-batch mode
  double* dalloc(size_t n) {
    dbufs.emplace_back(std::max<size_t>(n, 1));
    double* d = dbufs.back().get();
    B200_CUDA(cudaMemset(d, 0, std::max<size_t>(n, 1) * sizeof(double)));
    return d;
  }
  DevBuf<int> flagI, flagU, listI, listU, cnt, su, si, sj;
  DevBuf<float> sr;
  DevBuf<double> pow_out;
  std::vector<int> hs_u, hs_i, hs_j;
  std::vector<float> hs_r;
  long long samples_last = 0, cap_samples = 0, epoch_samples_override = 0;
  int shard_lo = 0, shard_hi = 0;  // device sampler draws users from [shard_lo, shard_hi) when set (multi-GPU user sharding)
  int grid = 0;
  // device-side replay of the glibc stream (glibc_*_kernel): pinned raw draws with the unread tail of the previous epoch in
  // front, their device copy, the jump tables, the consumed-draw counter
  bool glibc_device = true;
  int* h_raw = nullptr;            // pinned
  long long raw_cap = 0, raw_have = 0;  // capacity / draws currently in h_raw (all unread)
  DevBuf<int> d_raw, d_tables, d_consumed;
  long long tables_cap = 0;
  int hog_blocks = 8;  // hogwild CTAs per SM; a sharded (multi-GPU) run leaves room for the collective's CTAs
  // dataflow mode (mf_dataflow_kernel): dependency tables rebuilt from every epoch's sample stream
  bool dataflow = false;
  int df_grid = 0, bbits = 1, rbits = 1;
  DevBuf<int> applied, arrived, slot_prev, slot_expect, vals_a, vals_b;
  DevBuf<unsigned long long> keys_a, keys_b;
  DevBuf<unsigned char> sort_tmp;
  size_t sort_tmp_bytes = 0;
  DevBuf<float> inv1_b, inv2_b;
  std::vector<float> h_inv1, h_inv2;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  float* falloc(size_t n, const double* init) {
    fbufs.emplace_back(std::max<size_t>(n, 1));
    float* d = fbufs.back().get();
    if (init) {
      std::vector<float> tmp(n);
      for (size_t i = 0; i < n; ++i) tmp[i] = (float)init[i];
      B200_CUDA(cudaMemcpy(d, tmp.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    } else {
      B200_CUDA(cudaMemset(d, 0, std::max<size_t>(n, 1) * sizeof(float)));
    }
    return d;
  }
};

namespace {

const void* dataflow_kernel_for(bool bpr, int f) {
  const bool one4 = (f % 4) == 0 && f <= 128;
  if (bpr) return one4 ? (const void*)mf_dataflow_kernel<true, true> : (const void*)mf_dataflow_kernel<true, false>;
  return one4 ? (const void*)mf_dataflow_kernel<false, true> : (const void*)mf_dataflow_kernel<false, false>;
}

long long epoch_batches(const b200_mf_s* h) {
  // pyx:586 (BPR: n_users / batch_size + 1) and pyx:292 (FunkSVD: nnz / batch_size + 1)
  return (h->p.algorithm == MF_BPR ? (long long)h->p.n_users : h->nnz) / h->p.batch_size + 1;
}

void host_samples(b200_mf_s* h, long long n) {
  // sampleBPR_Cython pyx:943-987 / sampleMSE_Cython pyx:881-938, draw for draw
  h->hs_u.resize((size_t)n); h->hs_i.resize((size_t)n);
  if (h->p.algorithm == MF_BPR) h->hs_j.resize((size_t)n); else h->hs_r.resize((size_t)n);
  const int* indptr = h->h_indptr.data();
  const int* indices = h->h_indices.data();
  const int nU = h->p.n_users, nI = h->p.n_items;
  for (long long g = 0; g < n; ++g) {
    long u = 0, start = 0, len = 0;
    while (len == 0 || len == nI) {
      u = h->rng.next() % nU;
      start = indptr[u];
      len = indptr[u + 1] - start;
    }
    bool positive = true;
    if (h->p.algorithm == FUNK_SVD && h->quota != 0.0f) positive = h->rng.next() <= (double)h->quota * 2147483647.0;
    long item = -1;
    float r = 0.f;
    if (h->p.algorithm == MF_BPR || positive) {
      const long k = h->rng.next() % len;
      item = indices[start + k];
      if (h->p.algorithm == FUNK_SVD) r = h->h_data[(size_t)(start + k)];
    }
    if (h->p.algorithm == MF_BPR || !positive) {
      long neg;
      for (;;) {
        neg = h->rng.next() % nI;
        const int* lo = std::lower_bound(indices + start, indices + start + len, (int)neg);
        if (lo == indices + start + len || *lo != neg) break;
      }
      if (h->p.algorithm == MF_BPR) h->hs_j[(size_t)g] = (int)neg; else { item = neg; r = 0.f; }
    }
    h->hs_u[(size_t)g] = (int)u;
    h->hs_i[(size_t)g] = (int)item;
    if (h->p.algorithm == FUNK_SVD) h->hs_r[(size_t)g] = r;
  }
}


// The epoch's n samples from the glibc stream, resolved on the device (see glibc_len_kernel).  Synchronises the stream once
// (the host must know how many draws were consumed before it can continue the stream).
void glibc_device_samples(b200_mf_s* h, long long n, cudaStream_t st) {
  const Params& p = h->p;
  const int per = 3;  // draws of a sample without rejections (user, positive | quota, negative | item)
  int levels = 1;
  while ((1ll << levels) < n) ++levels;
  long long want = n * per + n / 16 + 4096;
  for (int attempt = 0;; ++attempt) {
    B200_REQUIRE(attempt < 8 && want < (1ll << 30), "b200_mf_epoch: the glibc replay buffer does not converge (degenerate URM?)");
    if (want > h->raw_cap) {
      int* fresh = nullptr;
      B200_CUDA(cudaMallocHost(reinterpret_cast<void**>(&fresh), sizeof(int) * (size_t)want));
      if (h->raw_have) memcpy(fresh, h->h_raw, sizeof(int) * (size_t)h->raw_have);
      if (h->h_raw) cudaFreeHost(h->h_raw);
      h->h_raw = fresh;
      h->raw_cap = want;
      h->d_raw.alloc((size_t)want);
    }
    for (long long q = h->raw_have; q < want; ++q) h->h_raw[q] = h->rng.next();
    h->raw_have = want;
    const int R = (int)want;
    if ((long long)levels * (R + 1) > h->tables_cap) {
      h->tables_cap = (long long)levels * (R + 1);
      h->d_tables.alloc((size_t)h->tables_cap);
    }
    if (h->d_consumed.n == 0) h->d_consumed.alloc(1);
    B200_CUDA(cudaMemcpyAsync(h->d_raw.get(), h->h_raw, sizeof(int) * (size_t)R, cudaMemcpyHostToDevice, st));
    B200_CUDA(cudaMemsetAsync(h->d_consumed.get(), 0, sizeof(int), st));
    GlibcView v{h->d_raw.get(), R, h->d_indptr.get(), h->d_indices.get(), h->d_data.get(), p.n_users, p.n_items, p.algorithm, h->quota};
    int* T = h->d_tables.get();
    glibc_len_kernel<<<div_up(R + 1, 256), 256, 0, st>>>(v, T);
    for (int k = 0; k + 1 < levels; ++k)
      glibc_double_kernel<<<div_up(R + 1, 256), 256, 0, st>>>(T + (size_t)k * (R + 1), R, T + (size_t)(k + 1) * (R + 1));
    glibc_emit_kernel<<<div_up(n, 256), 256, 0, st>>>(v, T, levels, n, h->su.get(), h->si.get(), h->sj.get(), h->sr.get(), h->d_consumed.get());
    B200_CUDA(cudaGetLastError());
    count_launch(levels + 1);
    int consumed = 0;
    B200_CUDA(cudaMemcpyAsync(&consumed, h->d_consumed.get(), sizeof(int), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    if (consumed != 0x7FFFFFFF && consumed <= R) {
      // the unread tail opens the next epoch's stream
      h->raw_have = R - consumed;
      if (h->raw_have) memmove(h->h_raw, h->h_raw + consumed, sizeof(int) * (size_t)h->raw_have);
      return;
    }
    want = want + want / 2;  // many rejections (dense profiles): a longer buffer, same draws in front
  }
}

}  // namespace

extern "C" {

int b200_mf_create(b200_mf_t* out, int64_t n_users, int64_t n_items, int64_t nnz, const int32_t* h_indptr,
                   const int32_t* h_indices, const float* h_data, int n_factors, int algorithm, int batch_size,
                   float negative_interactions_quota, float learning_rate, int use_bias, float user_reg, float item_reg,
                   float bias_reg, float positive_reg, float negative_reg, int sgd_mode, float gamma, float beta_1,
                   float beta_2, const double* h_user_factors, const double* h_item_factors, int has_seed,
                   uint32_t random_seed, int sampler, int hogwild) {
  if (out) *out = nullptr;
  b200_mf_s* h = nullptr;
  int rc = guarded([&] {
    B200_REQUIRE(out && h_indptr && h_user_factors && h_item_factors, "b200_mf_create: NULL argument");
    B200_REQUIRE(n_users > 0 && n_items > 0 && nnz >= 0 && nnz < (1ll << 31) - 1, "b200_mf_create: bad shape");
    B200_REQUIRE(n_factors >= 1 && batch_size >= 1, "b200_mf_create: n_factors and batch_size must be >= 1");
    B200_REQUIRE(algorithm == MF_BPR || algorithm == FUNK_SVD, "b200_mf_create: unknown algorithm %d", algorithm);
    B200_REQUIRE(sgd_mode >= SGD && sgd_mode <= ADAM, "b200_mf_create: unknown sgd_mode %d", sgd_mode);
    h = new b200_mf_s();
    Params& p = h->p;
    p.n_users = (int)n_users; p.n_items = (int)n_items; p.f = n_factors; p.batch_size = batch_size;
    p.algorithm = algorithm; p.use_bias = use_bias != 0; p.sgd_mode = sgd_mode; p.hogwild = hogwild != 0;
    p.lr = learning_rate; p.user_reg = user_reg; p.item_reg = item_reg; p.bias_reg = bias_reg;
    p.positive_reg = positive_reg; p.negative_reg = negative_reg;
    p.gamma = gamma; p.beta1 = beta_1; p.beta2 = beta_2;
    p.b1_pow = beta_1; p.b2_pow = beta_2;  // pyx:220-221
    h->nnz = nnz;
    h->quota = negative_interactions_quota;
    h->sampler = sampler;
    h->seed = has_seed ? random_seed : 1u;
    h->rng.seed(h->seed);
    if (const char* e = getenv("B200REC_GLIBC_HOST")) h->glibc_device = atoi(e) == 0;  // 1: the sequential host replay (A/B, tests)
    h->h_indptr.assign(h_indptr, h_indptr + n_users + 1);
    h->h_indices.assign(h_indices, h_indices + nnz);
    if (algorithm == FUNK_SVD) h->h_data.assign(h_data, h_data + nnz);
    h->d_indptr.alloc((size_t)n_users + 1);
    h->d_indices.alloc((size_t)std::max<int64_t>(nnz, 1));
    h->d_data.alloc((size_t)std::max<int64_t>(nnz, 1));
    B200_CUDA(cudaMemcpy(h->d_indptr.get(), h_indptr, sizeof(int) * ((size_t)n_users + 1), cudaMemcpyHostToDevice));
    if (nnz) {
      B200_CUDA(cudaMemcpy(h->d_indices.get(), h_indices, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice));
      B200_CUDA(cudaMemcpy(h->d_data.get(), h_data, sizeof(float) * (size_t)nnz, cudaMemcpyHostToDevice));
    }
    const size_t nUf = (size_t)n_users * n_factors, nIf = (size_t)n_items * n_factors;
    h->fbufs.reserve(40);
    p.U = h->falloc(nUf, h_user_factors);
    p.V = h->falloc(nIf, h_item_factors);
    h->dbufs.reserve(8);
    if (!p.hogwild) { p.accU = h->dalloc(nUf); p.accV = h->dalloc(nIf); }
    if (p.use_bias) {
      p.bu = h->falloc((size_t)n_users, nullptr); p.bi = h->falloc((size_t)n_items, nullptr); p.mu = h->falloc(1, nullptr);
      p.accbu = h->dalloc((size_t)n_users); p.accbi = h->dalloc((size_t)n_items); p.accmu = h->dalloc(1);
    }
    if (sgd_mode == ADAGRAD || sgd_mode == RMSPROP) {
      p.cU = h->falloc(nUf, nullptr); p.cV = h->falloc(nIf, nullptr);
      if (p.use_bias) { p.cbu = h->falloc((size_t)n_users, nullptr); p.cbi = h->falloc((size_t)n_items, nullptr); p.cmu = h->falloc(1, nullptr); }
    } else if (sgd_mode == ADAM) {
      p.m1U = h->falloc(nUf, nullptr); p.m2U = h->falloc(nUf, nullptr); p.m1V = h->falloc(nIf, nullptr); p.m2V = h->falloc(nIf, nullptr);
      if (p.use_bias) {
        p.m1bu = h->falloc((size_t)n_users, nullptr); p.m2bu = h->falloc((size_t)n_users, nullptr);
        p.m1bi = h->falloc((size_t)n_items, nullptr); p.m2bi = h->falloc((size_t)n_items, nullptr);
        p.m1mu = h->falloc(1, nullptr); p.m2mu = h->falloc(1, nullptr);
      }
    }
    h->flagI.alloc((size_t)n_items); h->flagU.alloc((size_t)n_users);
    h->listI.alloc((size_t)2 * batch_size); h->listU.alloc((size_t)batch_size); h->cnt.alloc(4);
    B200_CUDA(cudaMemset(h->flagI.get(), 0, sizeof(int) * (size_t)n_items));
    B200_CUDA(cudaMemset(h->flagU.get(), 0, sizeof(int) * (size_t)n_users));
    B200_CUDA(cudaMemset(h->cnt.get(), 0, sizeof(int) * 4));
    p.flagI = h->flagI.get(); p.flagU = h->flagU.get(); p.listI = h->listI.get(); p.listU = h->listU.get(); p.cnt = h->cnt.get();
    h->pow_out.alloc(2);
    p.pow_out = h->pow_out.get();
    h->cap_samples = epoch_batches(h) * batch_size;
    h->su.alloc((size_t)h->cap_samples); h->si.alloc((size_t)h->cap_samples);
    if (algorithm == MF_BPR) h->sj.alloc((size_t)h->cap_samples); else h->sr.alloc((size_t)h->cap_samples);
    p.su = h->su.get(); p.si = h->si.get(); p.sj = h->sj.get(); p.sr = h->sr.get();
    // cooperative grid: every block resident
    int per_sm = 0;
    const bool vec4 = (n_factors % 4) == 0;
    if (vec4) B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mf_epoch_kernel<true>, 256, 0));
    else B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mf_epoch_kernel<false>, 256, 0));
    B200_REQUIRE(per_sm >= 1, "b200_mf_create: epoch kernel does not fit on an SM");
    h->grid = sm_count() * std::min(per_sm, 8);
    // dataflow mode: the default for the mini-batch semantics without bias terms (the global bias is touched by every
    // sample, which turns the dependence chain into a barrier per batch: those runs keep the cooperative kernel);
    // B200REC_MF_DATAFLOW=0 selects the cooperative kernel for A/B runs
    {
      const char* e = getenv("B200REC_MF_DATAFLOW");
      h->dataflow = !p.hogwild && !p.use_bias && !(e && atoi(e) == 0);
    }
    if (h->dataflow) {
      const int S = algorithm == MF_BPR ? 3 : 2;
      const size_t rows = (size_t)n_users + (size_t)n_items, slots = (size_t)h->cap_samples * S;
      B200_REQUIRE(slots < (1ull << 31), "b200_mf_create: epoch too long for 32-bit slot ids");
      h->applied.alloc(rows); h->arrived.alloc(rows);
      B200_CUDA(cudaMemset(h->arrived.get(), 0, sizeof(int) * rows));
      h->slot_prev.alloc(slots); h->slot_expect.alloc(slots);
      h->keys_a.alloc(slots); h->keys_b.alloc(slots); h->vals_a.alloc(slots); h->vals_b.alloc(slots);
      const long long nb = epoch_batches(h);
      while ((1ll << h->bbits) < nb + 1) ++h->bbits;
      while ((1ull << h->rbits) < rows + 1) ++h->rbits;
      cub::DoubleBuffer<unsigned long long> dk(h->keys_a.get(), h->keys_b.get());
      cub::DoubleBuffer<int> dv(h->vals_a.get(), h->vals_b.get());
      B200_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, h->sort_tmp_bytes, dk, dv, (int)slots, 0, h->bbits + h->rbits));
      h->sort_tmp.alloc(h->sort_tmp_bytes + 16);
      if (sgd_mode == ADAM) { h->inv1_b.alloc((size_t)nb); h->inv2_b.alloc((size_t)nb); }
      p.applied = h->applied.get(); p.arrived = h->arrived.get();
      p.slot_prev = h->slot_prev.get(); p.slot_expect = h->slot_expect.get();
      p.inv1_b = h->inv1_b.get(); p.inv2_b = h->inv2_b.get();
      int per_sm_df = 0;
      B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_df, dataflow_kernel_for(algorithm == MF_BPR, n_factors), 256, 0));
      B200_REQUIRE(per_sm_df >= 1, "b200_mf_create: dataflow kernel does not fit on an SM");
      h->df_grid = sm_count() * std::min(per_sm_df, 8);
    }
    B200_CUDA(cudaEventCreate(&h->ev0));
    B200_CUDA(cudaEventCreate(&h->ev1));
    *out = h;
  });
  if (rc != B200_OK && h) delete h;
  return rc;
}

int b200_mf_destroy(b200_mf_t h) {
  if (!h) return B200_OK;
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->h_raw) cudaFreeHost(h->h_raw);
  delete h;
  return B200_OK;
}

int b200_mf_epoch(b200_mf_t h, void* stream) {
  return guarded([&] {
    B200_REQUIRE(h != nullptr, "b200_mf_epoch: NULL handle");
    cudaStream_t st = (cudaStream_t)stream;
    Params& p = h->p;
    p.n_batches = epoch_batches(h);
    if (h->epoch_samples_override > 0) p.n_batches = std::max<long long>(1, h->epoch_samples_override / p.batch_size);
    const long long n = p.n_batches * p.batch_size;
    if (h->sampler == 0 && h->glibc_device && n * 4 + 65536 < (1ll << 30)) {
      glibc_device_samples(h, n, st);
    } else if (h->sampler == 0) {
      host_samples(h, n);
      B200_CUDA(cudaMemcpyAsync(h->su.get(), h->hs_u.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
      B200_CUDA(cudaMemcpyAsync(h->si.get(), h->hs_i.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
      if (p.algorithm == MF_BPR) B200_CUDA(cudaMemcpyAsync(h->sj.get(), h->hs_j.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
      else B200_CUDA(cudaMemcpyAsync(h->sr.get(), h->hs_r.data(), sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, st));
    }
    B200_CUDA(cudaEventRecord(h->ev0, st));
    if (h->sampler != 0) {
      mf_sample_kernel<<<div_up(n, 256), 256, 0, st>>>(h->d_indptr.get(), h->d_indices.get(), h->d_data.get(), h->shard_lo,
                                                      (h->shard_hi > h->shard_lo ? h->shard_hi - h->shard_lo : p.n_users), p.n_items,
                                                      p.algorithm, h->quota, n, h->seed, h->epoch, h->su.get(), h->si.get(),
                                                      h->sj.get(), h->sr.get());
      count_launch();
    }
    if (p.hogwild) {
      mf_hogwild_kernel<<<sm_count() * h->hog_blocks, 256, 0, st>>>(p, n);
      B200_CUDA(cudaGetLastError());
      if (p.sgd_mode == ADAM) {  // powers advance once per size-1 batch
        p.b1_pow *= pow((double)p.beta1, (double)n);
        p.b2_pow *= pow((double)p.beta2, (double)n);
      }
    } else if (h->dataflow) {
      // dependency tables of this epoch's stream: (row, batch) keys sorted, run heads give hit counts and previous batches
      const bool bpr = p.algorithm == MF_BPR;
      const int S = bpr ? 3 : 2;
      const long long m = n * S;
      if (bpr) mf_slot_keys_kernel<true><<<div_up(n, 256), 256, 0, st>>>(p.su, p.si, p.sj, n, p.n_users, p.batch_size, h->bbits, h->keys_a.get(), h->vals_a.get());
      else mf_slot_keys_kernel<false><<<div_up(n, 256), 256, 0, st>>>(p.su, p.si, p.sj, n, p.n_users, p.batch_size, h->bbits, h->keys_a.get(), h->vals_a.get());
      count_launch();
      cub::DoubleBuffer<unsigned long long> dk(h->keys_a.get(), h->keys_b.get());
      cub::DoubleBuffer<int> dv(h->vals_a.get(), h->vals_b.get());
      size_t tb = h->sort_tmp_bytes;
      B200_CUDA(cub::DeviceRadixSort::SortPairs(h->sort_tmp.get(), tb, dk, dv, (int)m, 0, h->bbits + h->rbits, st));
      count_launch();
      mf_deps_kernel<<<div_up(m, 256), 256, 0, st>>>(dk.Current(), dv.Current(), m, h->bbits, h->slot_prev.get(), h->slot_expect.get());
      count_launch();
      B200_CUDA(cudaMemsetAsync(h->applied.get(), 0xFF, sizeof(int) * ((size_t)p.n_users + (size_t)p.n_items), st));  // -1
      if (p.sgd_mode == ADAM) {  // the powers advance once per batch (pyx:649-652), the same repeated product as the other kernel
        h->h_inv1.resize((size_t)p.n_batches); h->h_inv2.resize((size_t)p.n_batches);
        double b1p = p.b1_pow, b2p = p.b2_pow;
        for (long long b = 0; b < p.n_batches; ++b) {
          h->h_inv1[(size_t)b] = (float)(1.0 / (1.0 - b1p));
          h->h_inv2[(size_t)b] = (float)(1.0 / (1.0 - b2p));
          b1p *= (double)p.beta1; b2p *= (double)p.beta2;
        }
        B200_CUDA(cudaMemcpyAsync(h->inv1_b.get(), h->h_inv1.data(), sizeof(float) * (size_t)p.n_batches, cudaMemcpyHostToDevice, st));
        B200_CUDA(cudaMemcpyAsync(h->inv2_b.get(), h->h_inv2.data(), sizeof(float) * (size_t)p.n_batches, cudaMemcpyHostToDevice, st));
        p.b1_pow = b1p; p.b2_pow = b2p;
      }
      long long n_arg = n;
      void* args[] = {(void*)&p, (void*)&n_arg};
      // cooperative launch only for its co-residency guarantee (the progress argument needs every warp resident)
      B200_CUDA(cudaLaunchCooperativeKernel(dataflow_kernel_for(bpr, p.f), dim3(h->df_grid), dim3(256), args, 0, st));
    } else {
      void* args[] = {(void*)&p};
      if (p.f % 4 == 0) B200_CUDA(cudaLaunchCooperativeKernel((void*)mf_epoch_kernel<true>, dim3(h->grid), dim3(256), args, 0, st));
      else B200_CUDA(cudaLaunchCooperativeKernel((void*)mf_epoch_kernel<false>, dim3(h->grid), dim3(256), args, 0, st));
    }
    count_launch();
    B200_CUDA(cudaEventRecord(h->ev1, st));
    h->timed = true;
    if (h->dataflow && p.sgd_mode == ADAM) {
      B200_CUDA(cudaStreamSynchronize(st));  // the host-side inv tables are reused by the next epoch
    } else if (!p.hogwild && p.sgd_mode == ADAM) {
      double pw[2];
      B200_CUDA(cudaMemcpyAsync(pw, h->pow_out.get(), sizeof(pw), cudaMemcpyDeviceToHost, st));
      B200_CUDA(cudaStreamSynchronize(st));
      p.b1_pow = pw[0];
      p.b2_pow = pw[1];
    } else if (h->sampler == 0 && !(h->glibc_device && n * 4 + 65536 < (1ll << 30))) {
      B200_CUDA(cudaStreamSynchronize(st));  // the host sample vectors are reused by the next epoch
    }
    h->samples_last = n;
    h->epoch += 1;
  });
}

int b200_mf_set_user_shard(b200_mf_t h, int user_lo, int user_hi, int64_t samples_per_epoch, uint32_t stream_id) {
  return guarded([&] {
    B200_REQUIRE(h != nullptr, "b200_mf_set_user_shard: NULL handle");
    B200_REQUIRE(h->sampler != 0, "b200_mf_set_user_shard: only the device (Philox) sampler can be sharded");
    B200_REQUIRE(0 <= user_lo && user_lo < user_hi && user_hi <= h->p.n_users, "b200_mf_set_user_shard: bad range [%d,%d)", user_lo, user_hi);
    B200_REQUIRE(samples_per_epoch >= 0 && samples_per_epoch <= h->cap_samples, "b200_mf_set_user_shard: samples_per_epoch out of range");
    h->shard_lo = user_lo;
    h->shard_hi = user_hi;
    h->epoch_samples_override = samples_per_epoch;
    h->seed += 0x9E3779B9u * stream_id;  // decorrelates the ranks' Philox streams
    h->hog_blocks = 6;  // 1536 of an SM's 2048 threads: the all-reduce kernels of the overlapped exchange fit beside it
  });
}

int b200_mf_samples_last_epoch(b200_mf_t h, int64_t* n) {
  return guarded([&] {
    B200_REQUIRE(h && n, "b200_mf_samples_last_epoch: NULL argument");
    *n = h->samples_last;
  });
}

int b200_mf_get_samples(b200_mf_t h, int32_t* u, int32_t* i, int32_t* j, float* r) {
  return guarded([&] {
    B200_REQUIRE(h != nullptr, "b200_mf_get_samples: NULL handle");
    B200_CUDA(cudaDeviceSynchronize());
    const size_t n = (size_t)h->samples_last;
    if (u) B200_CUDA(cudaMemcpy(u, h->su.get(), sizeof(int) * n, cudaMemcpyDeviceToHost));
    if (i) B200_CUDA(cudaMemcpy(i, h->si.get(), sizeof(int) * n, cudaMemcpyDeviceToHost));
    if (j && h->p.algorithm == MF_BPR) B200_CUDA(cudaMemcpy(j, h->sj.get(), sizeof(int) * n, cudaMemcpyDeviceToHost));
    if (r && h->p.algorithm == FUNK_SVD) B200_CUDA(cudaMemcpy(r, h->sr.get(), sizeof(float) * n, cudaMemcpyDeviceToHost));
  });
}

int b200_mf_get_factors(b200_mf_t h, double* user_factors, double* item_factors, double* user_bias, double* item_bias,
                        double* global_bias) {
  return guarded([&] {
    B200_REQUIRE(h != nullptr, "b200_mf_get_factors: NULL handle");
    B200_CUDA(cudaDeviceSynchronize());
    auto fetch = [&](const float* d, double* out, size_t n) {
      if (!out || !d) return;
      std::vector<float> tmp(n);
      B200_CUDA(cudaMemcpy(tmp.data(), d, n * sizeof(float), cudaMemcpyDeviceToHost));
      for (size_t k = 0; k < n; ++k) out[k] = (double)tmp[k];
    };
    fetch(h->p.U, user_factors, (size_t)h->p.n_users * h->p.f);
    fetch(h->p.V, item_factors, (size_t)h->p.n_items * h->p.f);
    fetch(h->p.bu, user_bias, (size_t)h->p.n_users);
    fetch(h->p.bi, item_bias, (size_t)h->p.n_items);
    fetch(h->p.mu, global_bias, 1);
  });
}

int b200_mf_device_factors(b200_mf_t h, float** d_user_factors, float** d_item_factors) {
  return guarded([&] {
    B200_REQUIRE(h != nullptr, "b200_mf_device_factors: NULL handle");
    if (d_user_factors) *d_user_factors = h->p.U;
    if (d_item_factors) *d_item_factors = h->p.V;
  });
}

int b200_mf_delta_snapshot_device(const float* d_V, float* d_B, float* d_own, float* d_sum, int64_t n, void* stream) {
  return guarded([&] {
    B200_REQUIRE(d_V && d_B && d_own && d_sum && n >= 0 && (n & 3) == 0, "b200_mf_delta_snapshot_device: bad argument (n must be a multiple of 4)");
    if (n == 0) return;
    mf_delta_snapshot_kernel<<<sm_count() * 8, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(d_V), reinterpret_cast<float4*>(d_B),
                                                                             reinterpret_cast<float4*>(d_own), reinterpret_cast<float4*>(d_sum), n / 4);
    B200_CUDA(cudaGetLastError());
    count_launch();
  });
}

int b200_mf_delta_apply_device(float* d_V, float* d_B, const float* d_sum, const float* d_own, int64_t n, void* stream) {
  return guarded([&] {
    B200_REQUIRE(d_V && d_B && d_own && d_sum && n >= 0 && (n & 3) == 0, "b200_mf_delta_apply_device: bad argument (n must be a multiple of 4)");
    if (n == 0) return;
    mf_delta_apply_kernel<<<sm_count() * 8, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float4*>(d_V), reinterpret_cast<float4*>(d_B),
                                                                          reinterpret_cast<const float4*>(d_sum), reinterpret_cast<const float4*>(d_own), n / 4);
    B200_CUDA(cudaGetLastError());
    count_launch();
  });
}

int b200_mf_last_epoch_ms(b200_mf_t h, float* ms) {
  return guarded([&] {
    B200_REQUIRE(h && ms && h->timed, "b200_mf_last_epoch_ms: no epoch run yet");
    B200_CUDA(cudaEventSynchronize(h->ev1));
    B200_CUDA(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  });
}

}  // extern "C"
