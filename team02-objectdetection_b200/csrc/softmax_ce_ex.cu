// softmax_ce_ex.cu -- nn.CrossEntropyLoss with its options (weight, ignore_index, label_smoothing, reduction) and uint8
// targets: the three paths of softmax_ce.cu / generic_ops.cu (4 pixels per thread, one pixel per thread, any C) with the
// options as template bits and run-time values.  They live in a translation unit of their own: sharing one with the
// default kernels changed ptxas's instruction schedule of those, which must stay as measured.
//
// For a counted pixel (target t in [0,C) and t != ignore_index), with lse = logsumexp_c z_c, class weights w (1 without a
// weight tensor), Wsum = sum_c w_c and eps = label_smoothing:
//   loss      = (1-eps) w_t (lse - z_t) + eps/C sum_c w_c (lse - z_c)
//   d/dz_c    = (1-eps) w_t (p_c - [c=t]) + eps/C (Wsum p_c - w_c)          p = softmax(z)
// Every other pixel has loss 0 and gradient 0, except that a bad label (neither counted nor ignore_index) makes its loss
// NaN.  Logits are handled shifted by their maximum m: lse - z_c = log(sum) - (z_c - m), where z_c - m <= 0, so both terms
// of the smoothing sum Wsum log(sum) - sum_c w_c (z_c - m) are >= 0 for non-negative weights (no cancellation).
#include "common.cuh"

namespace b200 {

enum { CE_U8 = 1,      // uint8 targets (else int64)
       CE_MAP = 2 };   // per pixel: loss map (forward) or gradient scaled by gout (backward); else reduced into loss_sum

struct CeExParams {
  const float* logits;     // NCHW f32 [B,C,H,W]
  const void* target;      // [B,H,W] int64 | uint8
  const float* weight;     // f32 [C] or nullptr (all ones)
  const float* gout;       // CE_MAP backward: f32 [B,H,W] incoming gradient of the loss map
  const double* denom;     // reduction: the 'mean' divisor in denom[0] (gradient scale 1/denom[0]), or nullptr ('sum')
  double* loss_sum;        // reduction: += sum of the pixel losses
  float* loss_map;         // CE_MAP forward: f32 [B,H,W]
  float* dlogits;          // NCHW f32 gradient, or nullptr
  long long ignore_index;
  float eps;               // label_smoothing
  int B, C;
  long long HW;
};

__device__ __forceinline__ float ce_nan() { return __int_as_float(0x7fc00000); }

__device__ __forceinline__ bool ce_counted(long long t, int C, long long ignore_index) {
  return t >= 0 && t < C && t != ignore_index;
}

// loss of one pixel: ls = log(sum of exp(z - m)), zt = z_t - m, swz = sum_c w_c (z_c - m), k = eps / C
__device__ __forceinline__ float ce_ex_loss(bool counted, bool ignored, float wt, float ls, float zt, float swz, float wsum,
                                            float eps, float k) {
  if (!counted) return ignored ? 0.f : ce_nan();
  float l = (1.f - eps) * wt * (ls - zt);
  if (k != 0.f) l = fmaf(k, fmaf(wsum, ls, -swz), l);   // skipped without smoothing: a -inf logit would make it 0 * inf
  return l;
}

// target of pixel i as an integer
template <int MODE>
__device__ __forceinline__ long long ce_target(const void* target, long long i) {
  if constexpr ((MODE & CE_U8) != 0) return (long long)__ldg(reinterpret_cast<const uint8_t*>(target) + i);
  else return __ldg(reinterpret_cast<const long long*>(target) + i);
}

// d loss / d z_c of a counted pixel before the reduction scale: q = p_c, bt = (1-eps) w_t, k = eps / C.  As the two terms
// (1-eps) w_t (p_c - [c=t]) + k (Wsum p_c - w_c): each is exactly 0 where it should be (C = 1: p = 1, Wsum = w)
__device__ __forceinline__ float ce_ex_grad(float q, bool is_t, float bt, float k, float wsum, float wc) {
  return fmaf(bt, is_t ? q - 1.f : q, k * fmaf(wsum, q, -wc));
}

// block-wide (256 threads) sum of one float per thread, added to *out in f64 by one atomic per CTA
__device__ __forceinline__ void ce_block_sum_f64(float v, double* out) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __shared__ float wsum[8];
  if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 8) {
    float t = wsum[threadIdx.x];
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) t += __shfl_xor_sync(0xffu, t, o);
    if (threadIdx.x == 0) atomicAdd(out, (double)t);
  }
}

// denom[0] += sum of w_t over the counted pixels (the divisor of the weighted 'mean'); denom[1] += number of bad labels
// (neither counted nor ignore_index).  Accumulated in f64: the weighted partial sums are not integers.
template <typename TT>
__global__ void __launch_bounds__(256)
ce_count_ex_kernel(const TT* __restrict__ target, const float* __restrict__ weight, double* __restrict__ denom, long long N,
                   int C, long long ignore_index) {
  double d = 0.0, bad = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
    const long long t = (long long)__ldg(target + i);
    if (ce_counted(t, C, ignore_index)) d += weight ? (double)__ldg(weight + t) : 1.0;
    else if (t != ignore_index) bad += 1.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    d += __shfl_xor_sync(0xffffffffu, d, o);
    bad += __shfl_xor_sync(0xffffffffu, bad, o);
  }
  __shared__ double sd[8], sb[8];
  if ((threadIdx.x & 31) == 0) { sd[threadIdx.x >> 5] = d; sb[threadIdx.x >> 5] = bad; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double v = 0.0, b = 0.0;
    for (int i = 0; i < 8; ++i) { v += sd[i]; b += sb[i]; }
    if (v != 0.0) atomicAdd(denom, v);
    if (b != 0.0) atomicAdd(denom + 1, b);
  }
}

// Any class count (C > 32): three passes over the class planes (max and Wsum; sum of
// exp and sum w_c (z_c - m); loss and gradient), weights read through L1.
template <int MODE>
__global__ void __launch_bounds__(256)
softmax_ce_ex_generic_kernel(const CeExParams P) {
  constexpr bool MAP = (MODE & CE_MAP) != 0;
  const int C = P.C;
  const long long HW = P.HW;
  const long long total = (long long)P.B * HW;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float loss = 0.f;
  if (idx < total) {
    const int b = (int)(idx / HW);
    const long long pix = idx - (long long)b * HW;
    const float* lp = P.logits + (long long)b * C * HW + pix;
    const float* wp = P.weight;
    float m = -INFINITY, wsum = 0.f;
    for (int c = 0; c < C; ++c) {
      m = fmaxf(m, __ldg(lp + (long long)c * HW));
      wsum += wp ? __ldg(wp + c) : 1.f;
    }
    float sum = 0.f, swz = 0.f;
    for (int c = 0; c < C; ++c) {
      const float z = __ldg(lp + (long long)c * HW) - m;
      sum += expf(z);
      swz = fmaf(wp ? __ldg(wp + c) : 1.f, z, swz);
    }
    const long long t = ce_target<MODE>(P.target, idx);
    const bool counted = ce_counted(t, C, P.ignore_index);
    const float zt = counted ? __ldg(lp + t * HW) - m : 0.f;
    const float wt = counted ? (wp ? __ldg(wp + t) : 1.f) : 0.f;
    const float k = P.eps / (float)C;
    const float l = ce_ex_loss(counted, t == P.ignore_index, wt, logf(sum), zt, swz, wsum, P.eps, k);
    if constexpr (MAP) {
      if (P.loss_map) P.loss_map[idx] = l;
    } else {
      loss = l;
    }
    if (P.dlogits) {
      float gs;
      if constexpr (MAP) gs = __ldg(P.gout + idx);
      else gs = P.denom ? (float)(1.0 / __ldg(P.denom)) : 1.f;
      const float inv = 1.f / sum, bt = (1.f - P.eps) * wt;
      float* gp = P.dlogits + (long long)b * C * HW + pix;
      for (int c = 0; c < C; ++c) {
        const float q = expf(__ldg(lp + (long long)c * HW) - m) * inv;
        gp[(long long)c * HW] = counted ? ce_ex_grad(q, c == (int)t, bt, k, wsum, wp ? __ldg(wp + c) : 1.f) * gs : 0.f;
      }
    }
  }
  if constexpr (!MAP) ce_block_sum_f64(loss, P.loss_sum);
}

static int launch_softmax_ce_ex_generic(const CeExParams& p, int mode, cudaStream_t st) {
  const unsigned grid = (unsigned)(((long long)p.B * p.HW + 255) / 256);
  switch (mode) {
    case 0: softmax_ce_ex_generic_kernel<0><<<grid, 256, 0, st>>>(p); break;
    case CE_U8: softmax_ce_ex_generic_kernel<CE_U8><<<grid, 256, 0, st>>>(p); break;
    case CE_MAP: softmax_ce_ex_generic_kernel<CE_MAP><<<grid, 256, 0, st>>>(p); break;
    case CE_U8 | CE_MAP: softmax_ce_ex_generic_kernel<CE_U8 | CE_MAP><<<grid, 256, 0, st>>>(p); break;
    default: return set_error(-1, "softmax_ce_ex: bad mode %d", mode);
  }
  return check_launch("softmax_ce_ex");
}

// Register paths (C <= 32), selected by the conditions of b200seg_softmax_ce, with MODE = CE_U8 | CE_MAP as template bits.
// Class weights sit in registers (loaded once per thread from the device array; all ones when there is none); label
// smoothing and ignore_index are run-time values.
template <int CMAX, int MODE>
__global__ void __launch_bounds__(256)
softmax_ce_ex_kernel(const CeExParams P) {
  constexpr bool MAP = (MODE & CE_MAP) != 0;
  const int C = P.C;
  const long long HW = P.HW;
  const long long total = (long long)P.B * HW;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  float loss = 0.f;
  if (idx < total) {
    const int b = (int)(idx / HW);
    const long long pix = idx - (long long)b * HW;
    const float* lp = P.logits + (long long)b * C * HW + pix;
    float v[CMAX], w[CMAX];
    float m = -INFINITY, wsum = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      v[c] = (c < C) ? __ldg(lp + (long long)c * HW) : -INFINITY;
      w[c] = (c < C) ? (P.weight ? __ldg(P.weight + c) : 1.f) : 0.f;
      m = fmaxf(m, v[c]);
      wsum += w[c];
    }
    const long long t = ce_target<MODE>(P.target, idx);
    const bool counted = ce_counted(t, C, P.ignore_index);
    float sum = 0.f, zt = 0.f, wt = 0.f, swz = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      const float z = v[c] - m;
      if (c == (int)t) { zt = z; wt = w[c]; }
      if (c < C) swz = fmaf(w[c], z, swz);
      v[c] = (c < C) ? expf(z) : 0.f;
      sum += v[c];
    }
    const float k = P.eps / (float)C;
    const float l = ce_ex_loss(counted, t == P.ignore_index, wt, logf(sum), zt, swz, wsum, P.eps, k);
    if constexpr (MAP) {
      if (P.loss_map) P.loss_map[idx] = l;
    } else {
      loss = l;
    }
    if (P.dlogits) {
      float gs;
      if constexpr (MAP) gs = __ldg(P.gout + idx);
      else gs = P.denom ? (float)(1.0 / __ldg(P.denom)) : 1.f;
      const float inv = 1.f / sum, bt = (1.f - P.eps) * wt;
      float* gp = P.dlogits + (long long)b * C * HW + pix;
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < C) gp[(long long)c * HW] = counted ? ce_ex_grad(v[c] * inv, c == (int)t, bt, k, wsum, w[c]) * gs : 0.f;
    }
  }
  if constexpr (!MAP) ce_block_sum_f64(loss, P.loss_sum);
}

// Four consecutive pixels per thread (HW % 4 == 0): 16-byte class-plane loads and gradient stores as softmax_ce_x4_kernel;
// int64 targets in two 16-byte loads, uint8 targets in one 4-byte load; the loss map and gout as one float4 each.
template <int CMAX, int MODE>
__global__ void __launch_bounds__(256)
softmax_ce_ex_x4_kernel(const CeExParams P) {
  constexpr bool U8 = (MODE & CE_U8) != 0, MAP = (MODE & CE_MAP) != 0;
  const int C = P.C;
  const unsigned HW4 = (unsigned)(P.HW / 4);
  const unsigned total = (unsigned)P.B * HW4;           // groups of 4 pixels (launcher: < 2^31)
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
  float loss = 0.f;
  if (idx < total) {
    const unsigned b = idx / HW4, g = idx - b * HW4;
    const float4* lp = reinterpret_cast<const float4*>(P.logits) + (size_t)b * C * HW4 + g;
    float4 v[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
      v[c] = (c < C) ? __ldg(lp + (size_t)c * HW4) : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    long long tt[4];
    if constexpr (U8) {
      const uchar4 t4 = __ldg(reinterpret_cast<const uchar4*>(P.target) + idx);
      tt[0] = t4.x; tt[1] = t4.y; tt[2] = t4.z; tt[3] = t4.w;
    } else {
      const longlong2 t01 = __ldg(reinterpret_cast<const longlong2*>(P.target) + (size_t)idx * 2);
      const longlong2 t23 = __ldg(reinterpret_cast<const longlong2*>(P.target) + (size_t)idx * 2 + 1);
      tt[0] = t01.x; tt[1] = t01.y; tt[2] = t23.x; tt[3] = t23.y;
    }
    float w[CMAX], wsum = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      w[c] = (c < C) ? (P.weight ? __ldg(P.weight + c) : 1.f) : 0.f;
      wsum += w[c];
    }
    const float k = P.eps / (float)C;
    float inv[4], bt[4], l4[4];
    bool counted[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      float m = -INFINITY;
#pragma unroll
      for (int c = 0; c < CMAX; ++c) m = fmaxf(m, (&v[c].x)[p]);
      float sum = 0.f, zt = 0.f, wt = 0.f, swz = 0.f;
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        const float z = (&v[c].x)[p] - m;
        if (c == (int)tt[p]) { zt = z; wt = w[c]; }
        if (c < C) swz = fmaf(w[c], z, swz);
        const float e = (c < C) ? expf(z) : 0.f;
        (&v[c].x)[p] = e;
        sum += e;
      }
      counted[p] = ce_counted(tt[p], C, P.ignore_index);
      l4[p] = ce_ex_loss(counted[p], tt[p] == P.ignore_index, wt, logf(sum), zt, swz, wsum, P.eps, k);
      inv[p] = 1.f / sum;
      bt[p] = (1.f - P.eps) * wt;
    }
    if constexpr (MAP) {
      if (P.loss_map) reinterpret_cast<float4*>(P.loss_map)[idx] = make_float4(l4[0], l4[1], l4[2], l4[3]);
    } else {
      loss = (l4[0] + l4[1]) + (l4[2] + l4[3]);
    }
    if (P.dlogits) {
      float gs[4];
      if constexpr (MAP) {
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(P.gout) + idx);
        gs[0] = g4.x; gs[1] = g4.y; gs[2] = g4.z; gs[3] = g4.w;
      } else {
        const float s = P.denom ? (float)(1.0 / __ldg(P.denom)) : 1.f;
        gs[0] = gs[1] = gs[2] = gs[3] = s;
      }
      float4* gp = reinterpret_cast<float4*>(P.dlogits) + (size_t)b * C * HW4 + g;
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        if (c < C) {
          float4 o;
#pragma unroll
          for (int p = 0; p < 4; ++p)
            (&o.x)[p] = counted[p] ? ce_ex_grad((&v[c].x)[p] * inv[p], c == (int)tt[p], bt[p], k, wsum, w[c]) * gs[p] : 0.f;
          gp[(size_t)c * HW4] = o;
        }
      }
    }
  }
  if constexpr (!MAP) ce_block_sum_f64(loss, P.loss_sum);
}

template <int MODE>
static int launch_softmax_ce_ex(const CeExParams& P, cudaStream_t st) {
  constexpr bool U8 = (MODE & CE_U8) != 0;
  const long long total = (long long)P.B * P.HW;
  const uintptr_t tmask = U8 ? 3 : 15;
  const auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool aligned = P.HW % 4 == 0 && total / 4 < (1LL << 31) && al16(P.logits) &&
                       (reinterpret_cast<uintptr_t>(P.target) & tmask) == 0 && (!P.dlogits || al16(P.dlogits)) &&
                       (!P.loss_map || al16(P.loss_map)) && (!P.gout || al16(P.gout));
  if (P.C <= 16 && aligned) {
    const unsigned g4 = (unsigned)((total / 4 + 255) / 256);
    if (P.C <= 10) softmax_ce_ex_x4_kernel<10, MODE><<<g4, 256, 0, st>>>(P);
    else softmax_ce_ex_x4_kernel<16, MODE><<<g4, 256, 0, st>>>(P);
    return check_launch("softmax_ce_ex");
  }
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (P.C <= 16) softmax_ce_ex_kernel<16, MODE><<<grid, 256, 0, st>>>(P);
  else if (P.C <= 32) softmax_ce_ex_kernel<32, MODE><<<grid, 256, 0, st>>>(P);
  else return launch_softmax_ce_ex_generic(P, MODE, st);
  return check_launch("softmax_ce_ex");
}

static int dispatch_softmax_ce_ex(const CeExParams& P, bool u8, bool map, cudaStream_t st) {
  if (u8) return map ? launch_softmax_ce_ex<CE_U8 | CE_MAP>(P, st) : launch_softmax_ce_ex<CE_U8>(P, st);
  return map ? launch_softmax_ce_ex<CE_MAP>(P, st) : launch_softmax_ce_ex<0>(P, st);
}

}  // namespace b200

using namespace b200;

static int ce_ex_check(const float* logits, const void* target, int target_dtype, float label_smoothing, int B, int C, int H,
                       int W, const char* what) {
  B200_REQUIRE(C >= 1, "%s: C=%d", what, C);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "%s: empty tensor", what);
  B200_REQUIRE(logits && target, "%s: null logits / target", what);
  B200_REQUIRE(target_dtype == B200SEG_I64 || target_dtype == B200SEG_U8, "%s: target_dtype %d (B200SEG_I64 | B200SEG_U8)",
               what, target_dtype);
  B200_REQUIRE(label_smoothing >= 0.f && label_smoothing <= 1.f, "%s: label_smoothing %g not in [0, 1]", what,
               (double)label_smoothing);
  return 0;
}

extern "C" int b200seg_softmax_ce_ex(const float* logits, const void* target, int target_dtype, long long ignore_index,
                                     const float* weight, float label_smoothing, double* loss_sum, float* loss_map,
                                     float* dlogits, const double* denom, int B, int C, int H, int W, b200seg_stream_t s) {
  if (int rc = ce_ex_check(logits, target, target_dtype, label_smoothing, B, C, H, W, "softmax_ce_ex")) return rc;
  B200_REQUIRE((loss_sum != nullptr) != (loss_map != nullptr), "softmax_ce_ex: exactly one of loss_sum / loss_map");
  B200_REQUIRE(!(loss_map && dlogits), "softmax_ce_ex: the loss-map forward writes no gradient (b200seg_softmax_ce_ex_bwd)");
  B200_REQUIRE(!(loss_map && denom), "softmax_ce_ex: denom scales a reduced loss, not a loss map");
  CeExParams P{logits, target, weight, nullptr, denom, loss_sum, loss_map, dlogits, ignore_index, label_smoothing, B, C,
               (long long)H * W};
  return dispatch_softmax_ce_ex(P, target_dtype == B200SEG_U8, loss_map != nullptr, (cudaStream_t)s);
}

extern "C" int b200seg_softmax_ce_ex_bwd(const float* logits, const void* target, int target_dtype, long long ignore_index,
                                         const float* weight, float label_smoothing, const float* gout, float* dlogits, int B,
                                         int C, int H, int W, b200seg_stream_t s) {
  if (int rc = ce_ex_check(logits, target, target_dtype, label_smoothing, B, C, H, W, "softmax_ce_ex_bwd")) return rc;
  B200_REQUIRE(gout && dlogits, "softmax_ce_ex_bwd: null gout / dlogits");
  CeExParams P{logits, target, weight, gout, nullptr, nullptr, nullptr, dlogits, ignore_index, label_smoothing, B, C,
               (long long)H * W};
  return dispatch_softmax_ce_ex(P, target_dtype == B200SEG_U8, true, (cudaStream_t)s);
}

extern "C" int b200seg_ce_count_ex(const void* target, int target_dtype, long long ignore_index, const float* weight, double* denom,
                        long long N, int C, b200seg_stream_t s) {
  B200_REQUIRE(target && denom && N > 0 && C >= 1, "ce_count_ex: bad arguments");
  B200_REQUIRE(target_dtype == B200SEG_I64 || target_dtype == B200SEG_U8, "ce_count_ex: target_dtype %d (B200SEG_I64 | B200SEG_U8)",
               target_dtype);
  long long g = (N + 256 * 8 - 1) / (256 * 8);
  if (g > 148 * 8) g = 148 * 8;
  cudaStream_t st = (cudaStream_t)s;
  if (target_dtype == B200SEG_U8)
    ce_count_ex_kernel<uint8_t><<<(unsigned)g, 256, 0, st>>>((const uint8_t*)target, weight, denom, N, C, ignore_index);
  else
    ce_count_ex_kernel<long long><<<(unsigned)g, 256, 0, st>>>((const long long*)target, weight, denom, N, C, ignore_index);
  return check_launch("ce_count_ex");
}
