// seg_metrics.cu -- validation metrics over logits that already exist (SegmentationMetrics.update, the fp32 path, tails the
// fused kernel does not cover, and the plain UNet's NHWC logits buffer): confusion matrix, valid / invalid counts and the
// cross-entropy sum, accumulated per CTA in shared memory (seg_metrics.cuh) and flushed once per CTA.
//
// Three access patterns, one per-pixel rule:
//   nchw4    NCHW with H*W % 4 == 0: a thread owns 4 consecutive pixels and reads each class plane with one 16-byte (f32) or
//            8-byte (bf16) load, its 4 int64 targets with two 16-byte loads (uint8: one 4-byte load) -- as softmax_ce_x4
//   nhwc     NHWC with a 16-byte pixel pitch (UNet's logits, ldc = 16): a thread owns one pixel and reads it in 16-byte pieces
//   strided  anything else (odd W, unaligned views, odd ldc): one pixel per thread, scalar loads
// Grid-stride loops over one resident wave of CTAs, so the histogram is flushed ~600-1200 times per call, not once per tile.
#include "seg_metrics.cuh"

namespace b200 {

__device__ __forceinline__ long long seg_load_target(const void* tgt, bool u8, long long i) {
  return u8 ? (long long)__ldg(static_cast<const uint8_t*>(tgt) + i) : __ldg(static_cast<const long long*>(tgt) + i);
}

template <typename T>
__global__ void __launch_bounds__(256)
seg_metrics_nchw4_kernel(const T* __restrict__ lg, const void* __restrict__ tgt, bool u8, SegMetricsState ms, int B, int C,
                         unsigned HW4) {
  extern __shared__ uint32_t hist[];
  __shared__ uint32_t red[24];
  seg_hist_zero(hist, C);
  __syncthreads();
  float loss = 0.f;
  unsigned nvalid = 0, ninvalid = 0;
  const unsigned total = (unsigned)B * HW4;                 // B*H*W < 2^31 (launcher): 32-bit index arithmetic
  for (unsigned g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    const unsigned b = g / HW4, q = g - b * HW4;
    long long t[4];
    if (u8) {
      const uint32_t tv = __ldg(static_cast<const uint32_t*>(tgt) + g);
#pragma unroll
      for (int p = 0; p < 4; ++p) t[p] = (tv >> (8 * p)) & 0xff;
    } else {
      const longlong2 t01 = __ldg(static_cast<const longlong2*>(tgt) + 2 * g);
      const longlong2 t23 = __ldg(static_cast<const longlong2*>(tgt) + 2 * g + 1);
      t[0] = t01.x; t[1] = t01.y; t[2] = t23.x; t[3] = t23.y;
    }
    int tc[4];
    SegPix px[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) { tc[p] = seg_target_class(t[p], C, ms.ignore_index); seg_pix_init(px[p]); }
    const T* lp = lg + ((size_t)b * C * HW4 + q) * 4;
    for (int c = 0; c < C; ++c) {
      float v[4];
      if constexpr (sizeof(T) == 4) {
        const float4 f = __ldg(reinterpret_cast<const float4*>(lp + (size_t)c * HW4 * 4));
        v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
      } else {
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(lp + (size_t)c * HW4 * 4));
        v[0] = bf16lo(u.x); v[1] = bf16hi(u.x); v[2] = bf16lo(u.y); v[3] = bf16hi(u.y);
      }
#pragma unroll
      for (int p = 0; p < 4; ++p) seg_pix_step(px[p], v[p], c, tc[p]);
    }
#pragma unroll
    for (int p = 0; p < 4; ++p) seg_pix_finish(hist, px[p], t[p], tc[p], ms.ignore_index, C, loss, nvalid, ninvalid);
  }
  seg_flush(hist, C, loss, nvalid, ninvalid, red, ms);
}

// NHWC, ldc * sizeof(T) % 16 == 0, 16-byte aligned
template <typename T>
__global__ void __launch_bounds__(256)
seg_metrics_nhwc_kernel(const T* __restrict__ lg, int ldc, const void* __restrict__ tgt, bool u8, SegMetricsState ms,
                        long long P, int C) {
  extern __shared__ uint32_t hist[];
  __shared__ uint32_t red[24];
  seg_hist_zero(hist, C);
  __syncthreads();
  constexpr int VN = Vec16<T>::N;
  float loss = 0.f;
  unsigned nvalid = 0, ninvalid = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
    const long long t = seg_load_target(tgt, u8, i);
    const int tc = seg_target_class(t, C, ms.ignore_index);
    SegPix px;
    seg_pix_init(px);
    const T* lp = lg + i * ldc;
    for (int k = 0; k < C; k += VN) {
      Vec16<T> vec;
      vec.load(lp + k);
#pragma unroll
      for (int j = 0; j < VN; ++j)
        if (k + j < C) seg_pix_step(px, vec.v[j], k + j, tc);
    }
    seg_pix_finish(hist, px, t, tc, ms.ignore_index, C, loss, nvalid, ninvalid);
  }
  seg_flush(hist, C, loss, nvalid, ninvalid, red, ms);
}

// element (b, pixel p, class c) at lg[b * bstride + p * pstride + c * cstride]
template <typename T>
__global__ void __launch_bounds__(256)
seg_metrics_strided_kernel(const T* __restrict__ lg, long long bstride, long long pstride, long long cstride,
                           const void* __restrict__ tgt, bool u8, SegMetricsState ms, int B, int C, unsigned HW) {
  extern __shared__ uint32_t hist[];
  __shared__ uint32_t red[24];
  seg_hist_zero(hist, C);
  __syncthreads();
  float loss = 0.f;
  unsigned nvalid = 0, ninvalid = 0;
  const unsigned total = (unsigned)B * HW;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const unsigned b = i / HW, p = i - b * HW;
    const long long t = seg_load_target(tgt, u8, i);
    const int tc = seg_target_class(t, C, ms.ignore_index);
    SegPix px;
    seg_pix_init(px);
    const T* lp = lg + b * bstride + p * pstride;
    for (int c = 0; c < C; ++c, lp += cstride) seg_pix_step(px, to_f32<T>(*lp), c, tc);
    seg_pix_finish(hist, px, t, tc, ms.ignore_index, C, loss, nvalid, ninvalid);
  }
  seg_flush(hist, C, loss, nvalid, ninvalid, red, ms);
}

}  // namespace b200

using namespace b200;

extern "C" int b200seg_seg_metrics(const void* logits, int dtype, int layout, int ldc, const void* target, int target_dtype,
                                   long long ignore_index, int64_t* confusion, int64_t* counts, double* loss_sum, int B, int C,
                                   int H, int W, b200seg_stream_t s) {
  B200_REQUIRE(logits && target && confusion && counts && loss_sum, "seg_metrics: null pointer");
  B200_REQUIRE(C >= 1 && C <= 64, "seg_metrics: C=%d (1..64 classes: the confusion histogram lives in shared memory)", C);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "seg_metrics: empty tensor");
  B200_REQUIRE((long long)B * H * W < (1ll << 31), "seg_metrics: more than 2^31 - 1 pixels in one call");
  B200_REQUIRE(dtype == B200SEG_F32 || dtype == B200SEG_BF16, "seg_metrics: logits dtype must be f32 or bf16");
  B200_REQUIRE(target_dtype == B200SEG_I64 || target_dtype == B200SEG_U8, "seg_metrics: target dtype must be int64 or uint8");
  B200_REQUIRE(layout == B200SEG_NCHW || (layout == B200SEG_NHWC && ldc >= C), "seg_metrics: bad layout (%d) / ldc (%d)", layout, ldc);
  const bool u8 = target_dtype == B200SEG_U8;
  const bool bf = dtype == B200SEG_BF16;
  const int esz = bf ? 2 : 4;
  const long long HW = (long long)H * W, P = (long long)B * HW;
  const SegMetricsState ms{reinterpret_cast<unsigned long long*>(confusion), reinterpret_cast<unsigned long long*>(counts),
                           loss_sum, ignore_index};
  const size_t smem = (size_t)C * C * 4;
  const uintptr_t la = reinterpret_cast<uintptr_t>(logits), ta = reinterpret_cast<uintptr_t>(target);
  cudaStream_t st = (cudaStream_t)s;
  typedef __nv_bfloat16 bf16;
  // grid-stride over ONE resident wave (every CTA flushes its histogram once): CTAs per SM from the occupancy of the kernel
  // that is launched (registers and the C*C histogram decide it)
  auto launch = [&](auto kern, long long units, auto... kargs) -> int {
    int per_sm = 0;
    const cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, smem);
    if (e != cudaSuccess) return set_error((int)e, "seg_metrics: occupancy query: %s", cudaGetErrorString(e));
    const long long g = (units + 255) / 256, cap = (long long)sm_count() * (per_sm > 0 ? per_sm : 1);
    kern<<<(unsigned)(g < cap ? g : cap), 256, smem, st>>>(kargs...);
    return check_launch("seg_metrics");
  };
  if (layout == B200SEG_NCHW && HW % 4 == 0 && la % (4 * esz) == 0 && ta % (u8 ? 4 : 16) == 0) {
    if (bf) return launch(seg_metrics_nchw4_kernel<bf16>, P / 4, (const bf16*)logits, target, u8, ms, B, C, (unsigned)(HW / 4));
    return launch(seg_metrics_nchw4_kernel<float>, P / 4, (const float*)logits, target, u8, ms, B, C, (unsigned)(HW / 4));
  }
  if (layout == B200SEG_NHWC && ((long long)ldc * esz) % 16 == 0 && la % 16 == 0) {
    if (bf) return launch(seg_metrics_nhwc_kernel<bf16>, P, (const bf16*)logits, ldc, target, u8, ms, P, C);
    return launch(seg_metrics_nhwc_kernel<float>, P, (const float*)logits, ldc, target, u8, ms, P, C);
  }
  const long long bs = layout == B200SEG_NCHW ? C * HW : HW * ldc, ps = layout == B200SEG_NCHW ? 1 : ldc,
                  cs = layout == B200SEG_NCHW ? HW : 1;
  if (bf) return launch(seg_metrics_strided_kernel<bf16>, P, (const bf16*)logits, bs, ps, cs, target, u8, ms, B, C, (unsigned)HW);
  return launch(seg_metrics_strided_kernel<float>, P, (const float*)logits, bs, ps, cs, target, u8, ms, B, C, (unsigned)HW);
}
