// tail_fused.cu -- the output tail of MobileNetV2UNet.forward in ONE kernel (eval mode, bf16):
//
//     outc = outconv(32, C):  1x1 (32->16) + BN + ReLU -> 1x1 (16->C) + bias          (unet.py:108-121, :47)
//     final_upsample:         bilinear x2, align_corners=True                          (unet.py:30, :49)
//     [optional]              argmax over the classes -> uint8 mask                    (inference.py:64)
//     [optional]              validation metrics against targets: confusion histogram, valid / invalid counts and the
//                             cross-entropy sum (seg_metrics.cuh); no logits leave the chip
//
// Unfused these were three launches and two round trips of a 16/10-channel tensor through HBM (64 + 64 + 99 us at
// batch 64 on the B200: 0.32 / 0.48 / 0.36 of the HBM roofline).  Fused, the kernel reads the 32-channel decoder
// output once (64 B per half-resolution pixel) and writes the NCHW logits (or the mask) once; both 1x1 convs run on the
// tensor cores through warp-level mma.sync.m16n8k16 (K = 32 and K = 16 are far too small for a TMA/tcgen05 pipeline)
// with the hidden activation chained from the accumulator fragment of layer 1 into the A fragment of layer 2 in
// registers (bf16 rounding exactly where the unfused path stored it), and the half-resolution logits stay in shared
// memory in fp32 for the interpolation (the unfused path rounded them to bf16 first).
//
// Tile: one CTA = 32 x 128 output pixels.  align_corners=True maps output o to source o*(n-1)/(2n-1) < o/2, so the
// tile needs at most 18 x 66 source pixels; phase 1 computes their logits (16-pixel groups per warp, A fragments loaded
// straight from global: thread (g, t) of a group loads the 16-byte vector [8t, 8t+8) of pixels g and g+8 -- a fully
// coalesced 512-byte warp load -- and the K order of the weight fragments is permuted to match), phase 2 interpolates
// from shared memory with the same association as upsample2x_ac_kernel (vertical blend, then horizontal).
#include "seg_metrics.cuh"

namespace b200 {

constexpr int TAIL_TOH = 32, TAIL_TOW = 128;      // output tile
constexpr int TAIL_SR = 18, TAIL_SC = 66;         // source tile (rows, cols) incl. the +1 interpolation halo
constexpr int TAIL_NPX = TAIL_SR * TAIL_SC;       // 1188

__device__ __forceinline__ void tail_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t ld_pair(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const uint32_t*>(p)); }

// x   : NHWC bf16 [B,h,w,32]        w0 : bf16 [16][32] (BN folded)   b0 : f32 [16]
// w3  : bf16 [16][16] (rows >= C zero)   b3 : f32 [16]
// out : NCHW [B,C,2h,2w] of TO, or mask uint8 [B,2h,2w]
// TGT : void, or the target type (int64_t | uint8_t) of the metrics epilogue (tgt [B,2h,2w], state ms; out / mask unused)
template <typename TGT>
__device__ __forceinline__ void tail_metrics_phase2(const float* lg, uint32_t* hist, const TGT* __restrict__ tgt, const SegMetricsState& ms,
                                                    int b, int h, int w, int C, int oy0, int ox0, int yf, int xf, float sch,
                                                    float scw);

template <typename TO, bool ARGMAX, typename TGT = void>
__global__ void __launch_bounds__(256)
tail_fused_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w0, const float* __restrict__ b0,
                  const __nv_bfloat16* __restrict__ w3, const float* __restrict__ b3, TO* __restrict__ out,
                  uint8_t* __restrict__ mask, int B, int h, int w, int C, int tiles_x, int tiles_y,
                  const void* __restrict__ tgt, SegMetricsState ms) {
  constexpr bool METRICS = !std::is_void<TGT>::value;
  extern __shared__ float lg[];                   // [C][TAIL_NPX] half-resolution logits of this tile, fp32
                                                  // (metrics: then the u32 [C][C] histogram and 24 reduction words)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int Ho = 2 * h, Wo = 2 * w;
  int tile = blockIdx.x;
  const int txi = tile % tiles_x; tile /= tiles_x;
  const int tyi = tile % tiles_y;
  const int b = tile / tiles_y;
  const int oy0 = tyi * TAIL_TOH, ox0 = txi * TAIL_TOW;
  const float sch = (Ho > 1) ? (float)(h - 1) / (float)(Ho - 1) : 0.f;
  const float scw = (Wo > 1) ? (float)(w - 1) / (float)(Wo - 1) : 0.f;
  const int yf = (int)(sch * oy0), xf = (int)(scw * ox0);       // first source row / column of the tile

  // ---- weight fragments (held in registers for the whole CTA) ----
  // layer 1, K = 32 input channels in two k-steps; logical k of step s: slot 2t+j <-> channel 8t+4s+j, slot 2t+8+j <-> 8t+4s+2+j
  uint32_t bw0[2][2][2];                          // [k-step][n-tile][b0|b1]
#pragma unroll
  for (int s = 0; s < 2; ++s)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const __nv_bfloat16* row = w0 + (j * 8 + g) * 32 + 8 * t + 4 * s;
      bw0[s][j][0] = ld_pair(row);
      bw0[s][j][1] = ld_pair(row + 2);
    }
  // layer 2, K = 16 hidden channels in their natural order (the A fragment is layer 1's accumulator fragment)
  uint32_t bw3[2][2];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const __nv_bfloat16* row = w3 + (j * 8 + g) * 16 + 2 * t;
    bw3[j][0] = ld_pair(row);
    bw3[j][1] = ld_pair(row + 8);
  }
  float bias0[2][2], bias3[2][2];
#pragma unroll
  for (int j = 0; j < 2; ++j)
#pragma unroll
    for (int e = 0; e < 2; ++e) { bias0[j][e] = __ldg(b0 + j * 8 + 2 * t + e); bias3[j][e] = __ldg(b3 + j * 8 + 2 * t + e); }

  if constexpr (METRICS) seg_hist_zero(reinterpret_cast<uint32_t*>(lg + C * TAIL_NPX), C);   // published by phase 1's barrier

  // ---- phase 1: logits of the TAIL_SR x TAIL_SC source pixels ----
  const __nv_bfloat16* xb = x + (long long)b * h * w * 32;
  for (int grp = warp; grp < (TAIL_NPX + 15) / 16; grp += 8) {
    uint32_t a[2][4];                             // [k-step][a0..a3]
    int pidx[2];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const int i = grp * 16 + g + rr * 8;
      pidx[rr] = i;
      const int ty = i / TAIL_SC, tx = i - ty * TAIL_SC;
      const int gy = min(yf + ty, h - 1), gx = min(xf + tx, w - 1);      // clamped duplicates are never read in phase 2
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(xb + ((long long)gy * w + gx) * 32 + 8 * t));
      a[0][rr] = v.x; a[0][2 + rr] = v.y;         // step 0: channels 8t..8t+1 | 8t+2..8t+3
      a[1][rr] = v.z; a[1][2 + rr] = v.w;         // step 1: channels 8t+4..5  | 8t+6..7
    }
    float hacc[2][4];
#pragma unroll
    for (int j = 0; j < 2; ++j) { hacc[j][0] = bias0[j][0]; hacc[j][1] = bias0[j][1]; hacc[j][2] = bias0[j][0]; hacc[j][3] = bias0[j][1]; }
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
      for (int j = 0; j < 2; ++j) tail_mma(hacc[j], a[s], bw0[s][j][0], bw0[s][j][1]);
    // ReLU, round to bf16 (where the unfused path stored the hidden activation), re-use as layer 2's A fragment
    uint32_t ha[4];
    ha[0] = pack_bf16x2(fmaxf(hacc[0][0], 0.f), fmaxf(hacc[0][1], 0.f));
    ha[1] = pack_bf16x2(fmaxf(hacc[0][2], 0.f), fmaxf(hacc[0][3], 0.f));
    ha[2] = pack_bf16x2(fmaxf(hacc[1][0], 0.f), fmaxf(hacc[1][1], 0.f));
    ha[3] = pack_bf16x2(fmaxf(hacc[1][2], 0.f), fmaxf(hacc[1][3], 0.f));
    float lacc[2][4];
#pragma unroll
    for (int j = 0; j < 2; ++j) { lacc[j][0] = bias3[j][0]; lacc[j][1] = bias3[j][1]; lacc[j][2] = bias3[j][0]; lacc[j][3] = bias3[j][1]; }
#pragma unroll
    for (int j = 0; j < 2; ++j) tail_mma(lacc[j], ha, bw3[j][0], bw3[j][1]);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = j * 8 + 2 * t + e;
        if (c < C) {
          if (pidx[0] < TAIL_NPX) lg[c * TAIL_NPX + pidx[0]] = lacc[j][e];
          if (pidx[1] < TAIL_NPX) lg[c * TAIL_NPX + pidx[1]] = lacc[j][2 + e];
        }
      }
  }
  __syncthreads();

  if constexpr (METRICS) {
    tail_metrics_phase2<TGT>(lg, reinterpret_cast<uint32_t*>(lg + C * TAIL_NPX), static_cast<const TGT*>(tgt), ms, b, h, w, C,
                             oy0, ox0, yf, xf, sch, scw);
    return;
  }

  // ---- phase 2: bilinear x2 (align_corners=True) from shared memory; thread = 2 consecutive output pixels ----
  const int pr = threadIdx.x & 63, rq = threadIdx.x >> 6;
  const int ox = ox0 + 2 * pr;
  if (ox >= Wo) return;
  // the two outputs of a thread read source columns x0(ox), x0(ox)+1 and x0(ox+1), x0(ox+1)+1 with x0(ox+1) - x0(ox) in {0,1}:
  // three columns c0, c0+1, c0+2 cover both (a column past the right image border only ever gets weight 0)
  float lx[2];
  int d1;                                          // x0(ox+1) - x0(ox)
  int c0;
  {
    const float sx0 = scw * ox, sx1 = scw * (ox + 1);
    const int x0 = (int)sx0, x1 = (int)sx1;
    lx[0] = sx0 - x0; lx[1] = sx1 - x1;
    d1 = x1 - x0;
    c0 = x0 - xf;
  }
  const int ca = c0, cb = min(c0 + 1, TAIL_SC - 1), cc = min(c0 + 2, TAIL_SC - 1);
  for (int ry = rq; ry < TAIL_TOH; ry += 4) {
    const int oy = oy0 + ry;
    if (oy >= Ho) break;
    const float sy = sch * oy;
    const int y0 = (int)sy;
    const float ly = sy - y0, hy = 1.f - ly;
    const int r0 = (y0 - yf) * TAIL_SC, r1 = r0 + (y0 < h - 1 ? TAIL_SC : 0);
    float best[2] = {-INFINITY, -INFINITY};
    int bi[2] = {0, 0};
    for (int c = 0; c < C; ++c) {
      const float* pl = lg + c * TAIL_NPX;
      const float va = hy * pl[r0 + ca] + ly * pl[r1 + ca];
      const float vb = hy * pl[r0 + cb] + ly * pl[r1 + cb];
      const float vc = hy * pl[r0 + cc] + ly * pl[r1 + cc];
      float v[2];
      v[0] = (1.f - lx[0]) * va + lx[0] * vb;
      v[1] = (1.f - lx[1]) * (d1 ? vb : va) + lx[1] * (d1 ? vc : vb);
      if (ARGMAX) {
#pragma unroll
        for (int e = 0; e < 2; ++e)
          if (v[e] > best[e]) { best[e] = v[e]; bi[e] = c; }          // first maximum wins, like torch.max
      } else {
        TO* op = out + (((long long)b * C + c) * Ho + oy) * Wo + ox;
        if (sizeof(TO) == 2) *reinterpret_cast<uint32_t*>(op) = pack_bf16x2(v[0], v[1]);
        else *reinterpret_cast<float2*>(op) = make_float2(v[0], v[1]);
      }
    }
    if (ARGMAX) *reinterpret_cast<uint16_t*>(mask + ((long long)b * Ho + oy) * Wo + ox) = (uint16_t)(bi[0] | (bi[1] << 8));
  }
}

// Phase 2 of the metrics epilogue: the thread / pixel mapping and the interpolation arithmetic of the argmax epilogue above
// (so the predictions are the mask's, bit for bit), then log-sum-exp and the target logit over the same values.  No thread
// returns early: the flush at the end is a CTA barrier.
template <typename TGT>
__device__ __forceinline__ void tail_metrics_phase2(const float* lg, uint32_t* hist, const TGT* __restrict__ tgt,
                                                    const SegMetricsState& ms, int b, int h, int w, int C, int oy0, int ox0,
                                                    int yf, int xf, float sch, float scw) {
  const int Ho = 2 * h, Wo = 2 * w;
  const int pr = threadIdx.x & 63, rq = threadIdx.x >> 6;
  const int ox = ox0 + 2 * pr;
  float loss = 0.f;
  unsigned nvalid = 0, ninvalid = 0;
  if (ox < Wo) {
    float lx[2];
    int d1, c0;
    {
      const float sx0 = scw * ox, sx1 = scw * (ox + 1);
      const int x0 = (int)sx0, x1 = (int)sx1;
      lx[0] = sx0 - x0; lx[1] = sx1 - x1;
      d1 = x1 - x0;
      c0 = x0 - xf;
    }
    const int ca = c0, cb = min(c0 + 1, TAIL_SC - 1), cc = min(c0 + 2, TAIL_SC - 1);
    for (int ry = rq; ry < TAIL_TOH; ry += 4) {
      const int oy = oy0 + ry;
      if (oy >= Ho) break;
      // the two targets of the pixel pair: one 16-byte (int64) or 2-byte (uint8) load; Wo and ox are even
      long long t[2];
      const long long o = ((long long)b * Ho + oy) * Wo + ox;
      if constexpr (sizeof(TGT) == 8) {
        const longlong2 tv = __ldg(reinterpret_cast<const longlong2*>(tgt + o));
        t[0] = tv.x; t[1] = tv.y;
      } else {
        const unsigned short tv = __ldg(reinterpret_cast<const unsigned short*>(tgt + o));
        t[0] = tv & 0xff; t[1] = tv >> 8;
      }
      const int tc[2] = {seg_target_class(t[0], C, ms.ignore_index), seg_target_class(t[1], C, ms.ignore_index)};
      const float sy = sch * oy;
      const int y0 = (int)sy;
      const float ly = sy - y0, hy = 1.f - ly;
      const int r0 = (y0 - yf) * TAIL_SC, r1 = r0 + (y0 < h - 1 ? TAIL_SC : 0);
      SegPix px[2];
      seg_pix_init(px[0]); seg_pix_init(px[1]);
      for (int c = 0; c < C; ++c) {
        const float* pl = lg + c * TAIL_NPX;
        const float va = hy * pl[r0 + ca] + ly * pl[r1 + ca];
        const float vb = hy * pl[r0 + cb] + ly * pl[r1 + cb];
        const float vc = hy * pl[r0 + cc] + ly * pl[r1 + cc];
        float v[2];
        v[0] = (1.f - lx[0]) * va + lx[0] * vb;
        v[1] = (1.f - lx[1]) * (d1 ? vb : va) + lx[1] * (d1 ? vc : vb);
        seg_pix_step(px[0], v[0], c, tc[0]);
        seg_pix_step(px[1], v[1], c, tc[1]);
      }
#pragma unroll
      for (int e = 0; e < 2; ++e) seg_pix_finish(hist, px[e], t[e], tc[e], ms.ignore_index, C, loss, nvalid, ninvalid);
    }
  }
  seg_flush(hist, C, loss, nvalid, ninvalid, hist + C * C, ms);
}

}  // namespace b200

using namespace b200;

extern "C" int b200seg_tail_fused(const void* x, const void* w0, const float* b0, const void* w3, const float* b3, void* out,
                                  int out_dtype, uint8_t* mask, int B, int h, int w, int C, b200seg_stream_t s) {
  B200_REQUIRE(x && w0 && b0 && w3 && b3 && ((out != nullptr) != (mask != nullptr)), "tail_fused: bad pointers");
  B200_REQUIRE(C >= 1 && C <= 16 && B > 0 && h > 0 && w > 0, "tail_fused: bad shape (C=%d)", C);
  const int tiles_x = (2 * w + TAIL_TOW - 1) / TAIL_TOW, tiles_y = (2 * h + TAIL_TOH - 1) / TAIL_TOH;
  const long long grid = (long long)B * tiles_x * tiles_y;
  B200_REQUIRE(grid < (1ll << 31), "tail_fused: too many tiles");
  const size_t smem = (size_t)C * TAIL_NPX * sizeof(float);
  cudaStream_t st = (cudaStream_t)s;
  typedef __nv_bfloat16 bf16;
#define TAIL_LAUNCH(TO, AM)                                                                                            \
  {                                                                                                                    \
    static bool attr = false;                                                                                          \
    if (!attr) {                                                                                                       \
      cudaError_t e = cudaFuncSetAttribute(tail_fused_kernel<TO, AM>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * TAIL_NPX * 4); \
      if (e != cudaSuccess) return set_error((int)e, "tail_fused: cudaFuncSetAttribute: %s", cudaGetErrorString(e));   \
      attr = true;                                                                                                     \
    }                                                                                                                  \
    tail_fused_kernel<TO, AM><<<(unsigned)grid, 256, smem, st>>>((const bf16*)x, (const bf16*)w0, b0, (const bf16*)w3, b3, \
                                                                 (TO*)out, mask, B, h, w, C, tiles_x, tiles_y, nullptr, \
                                                                 SegMetricsState{});                                   \
  }
  if (mask) TAIL_LAUNCH(float, true)
  else if (out_dtype == B200SEG_BF16) TAIL_LAUNCH(bf16, false)
  else if (out_dtype == B200SEG_F32) TAIL_LAUNCH(float, false)
  else return set_error(-1, "tail_fused: bad out dtype");
#undef TAIL_LAUNCH
  return check_launch("tail_fused");
}

extern "C" int b200seg_tail_fused_metrics(const void* x, const void* w0, const float* b0, const void* w3, const float* b3,
                                          const void* target, int target_dtype, long long ignore_index, int64_t* confusion,
                                          int64_t* counts, double* loss_sum, int B, int h, int w, int C, b200seg_stream_t s) {
  B200_REQUIRE(x && w0 && b0 && w3 && b3 && target && confusion && counts && loss_sum, "tail_fused_metrics: bad pointers");
  B200_REQUIRE(C >= 1 && C <= 16 && B > 0 && h > 0 && w > 0, "tail_fused_metrics: bad shape (C=%d)", C);
  B200_REQUIRE(target_dtype == B200SEG_I64 || target_dtype == B200SEG_U8, "tail_fused_metrics: target dtype must be int64 or uint8");
  B200_REQUIRE((reinterpret_cast<uintptr_t>(target) & (target_dtype == B200SEG_I64 ? 15 : 1)) == 0,
               "tail_fused_metrics: target must be %d-byte aligned", target_dtype == B200SEG_I64 ? 16 : 2);
  const int tiles_x = (2 * w + TAIL_TOW - 1) / TAIL_TOW, tiles_y = (2 * h + TAIL_TOH - 1) / TAIL_TOH;
  const long long grid = (long long)B * tiles_x * tiles_y;
  B200_REQUIRE(grid < (1ll << 31), "tail_fused_metrics: too many tiles");
  const size_t smem = ((size_t)C * TAIL_NPX + C * C + 24) * 4;
  const SegMetricsState ms{reinterpret_cast<unsigned long long*>(confusion), reinterpret_cast<unsigned long long*>(counts),
                           loss_sum, ignore_index};
  cudaStream_t st = (cudaStream_t)s;
  typedef __nv_bfloat16 bf16;
#define TAIL_METRICS_LAUNCH(TGT)                                                                                       \
  {                                                                                                                    \
    static bool attr = false;                                                                                          \
    if (!attr) {                                                                                                       \
      cudaError_t e = cudaFuncSetAttribute(tail_fused_kernel<float, false, TGT>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           (16 * TAIL_NPX + 16 * 16 + 24) * 4);                                        \
      if (e != cudaSuccess) return set_error((int)e, "tail_fused_metrics: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); \
      attr = true;                                                                                                     \
    }                                                                                                                  \
    tail_fused_kernel<float, false, TGT><<<(unsigned)grid, 256, smem, st>>>((const bf16*)x, (const bf16*)w0, b0,        \
        (const bf16*)w3, b3, nullptr, nullptr, B, h, w, C, tiles_x, tiles_y, target, ms);                               \
  }
  if (target_dtype == B200SEG_I64) TAIL_METRICS_LAUNCH(int64_t)
  else TAIL_METRICS_LAUNCH(uint8_t)
#undef TAIL_METRICS_LAUNCH
  return check_launch("tail_fused_metrics");
}
