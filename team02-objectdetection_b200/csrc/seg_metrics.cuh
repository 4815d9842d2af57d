// seg_metrics.cuh -- per-pixel validation metrics shared by the fused output tail (tail_fused.cu) and the standalone
// kernels on existing logits (seg_metrics.cu): argmax, log-sum-exp, target logit, a per-CTA confusion histogram in
// shared memory and one flush per CTA into the caller's 64-bit state.
//
// Per pixel the classes are visited once, in order, with an online log-sum-exp: the running maximum m, its class and
// s = sum_c exp(z_c - m).  The maximum is replaced only on a strictly larger logit, so the first maximum wins (the rule
// of torch.argmax and of every argmax kernel in this library), and ties in the loss are exact: exp(0) = 1.
#pragma once
#include <cfloat>
#include <type_traits>

#include "common.cuh"

namespace b200 {

struct SegMetricsState {
  unsigned long long* confusion;   // [C][C], row = target, column = prediction
  unsigned long long* counts;      // [valid, invalid]
  double* loss_sum;                // sum over valid pixels of logsumexp(z) - z[target]
  long long ignore_index;
};

struct SegPix {
  float m, s, zt;
  int bi;
};

// The running maximum starts at -FLT_MAX, not -inf: a logit of -inf (a class masked out of logits handed to update()) then
// gives exp(-inf - m) = 0 even before the first finite class, where -inf - -inf would make the sum NaN.  A guard per class
// costs the issue-bound fused epilogue 23 us of 162 at batch 64.  Only a pixel whose logits are all <= -FLT_MAX keeps
// class 0 as its prediction where torch.argmax would name the first -FLT_MAX.
__device__ __forceinline__ void seg_pix_init(SegPix& p) { p.m = -FLT_MAX; p.s = 0.f; p.zt = 0.f; p.bi = 0; }

// one class logit v of class c; tc = the pixel's target class, or -1
__device__ __forceinline__ void seg_pix_step(SegPix& p, float v, int c, int tc) {
  const bool gt = v > p.m;
  const float e = expf(gt ? p.m - v : v - p.m);    // one exp either way (exp(-FLT_MAX - v) = 0 on the first class)
  p.s = gt ? fmaf(p.s, e, 1.f) : p.s + e;
  p.m = gt ? v : p.m;
  p.bi = gt ? c : p.bi;
  if (c == tc) p.zt = v;
}

// the pixel's target as a class index in [0, C), or -1 when it is out of range or ignore_index (which may be a class index:
// those pixels contribute nothing, as with nn.CrossEntropyLoss(ignore_index=k))
__device__ __forceinline__ int seg_target_class(long long t, int C, long long ignore_index) {
  return (t >= 0 && t < C && t != ignore_index) ? (int)t : -1;
}

// histogram bin of every lane that calls this (warp-aggregated: lanes with equal keys add once); key < 0 adds nothing
__device__ __forceinline__ void seg_hist_add(uint32_t* hist, int key) {
  const unsigned peers = __match_any_sync(__activemask(), key);
  if (key >= 0 && (__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(hist + key, (uint32_t)__popc(peers));
}

// finish one pixel: histogram, valid / invalid counters, loss partial
__device__ __forceinline__ void seg_pix_finish(uint32_t* hist, const SegPix& p, long long t, int tc, long long ignore_index,
                                               int C, float& loss, unsigned& nvalid, unsigned& ninvalid) {
  if (tc >= 0) {
    loss += (p.m - p.zt) + logf(p.s);
    ++nvalid;
  } else if (t != ignore_index) {
    ++ninvalid;
  }
  seg_hist_add(hist, tc >= 0 ? tc * C + p.bi : -1);
}

// Block-wide (256 threads) flush of the CTA's histogram and partials.  Every thread of the CTA calls it once; `red` is
// 24 words of shared memory.  Only nonzero bins and counters touch global memory.
__device__ __forceinline__ void seg_flush(const uint32_t* hist, int C, float loss, unsigned nvalid, unsigned ninvalid,
                                          uint32_t* red, const SegMetricsState& st) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    loss += __shfl_xor_sync(0xffffffffu, loss, o);
    nvalid += __shfl_xor_sync(0xffffffffu, nvalid, o);
    ninvalid += __shfl_xor_sync(0xffffffffu, ninvalid, o);
  }
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { red[warp] = __float_as_uint(loss); red[8 + warp] = nvalid; red[16 + warp] = ninvalid; }
  __syncthreads();                                 // also publishes the histogram
  for (int i = threadIdx.x; i < C * C; i += blockDim.x)
    if (hist[i]) atomicAdd(st.confusion + i, (unsigned long long)hist[i]);
  if (threadIdx.x == 0) {
    double l = 0.0;
    unsigned long long v = 0, bad = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { l += (double)__uint_as_float(red[i]); v += red[8 + i]; bad += red[16 + i]; }
    if (v) { atomicAdd(st.counts, v); atomicAdd(st.loss_sum, l); }
    if (bad) atomicAdd(st.counts + 1, bad);
  }
}

__device__ __forceinline__ void seg_hist_zero(uint32_t* hist, int C) {
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) hist[i] = 0;
}

}  // namespace b200
