// hbm_ops.cu -- the memory-bound operators: every kernel here moves each activation byte once,
// with 16-byte vector accesses that are contiguous along the NHWC channel axis.
//
//   conv3x3_smallcin   stem / UNet.inc conv0   (NCHW in -> NHWC out, folded BN + act)
//   dwconv3x3          depthwise 3x3 s1|s2     (folded BN + ReLU6)
//   upsample2x_concat  bilinear x2 (align_corners=False) fused with cat([skip, up])
//   upsample2x_ac_*    final bilinear x2 (align_corners=True) -> NCHW logits, or fused argmax mask
//   nhwc_to_nchw, maxpool2x2
#include <stdlib.h>

#include "common.cuh"

namespace b200 {

static inline int grid_for(long long items, int threads) {
  if (items >= (1LL << 31)) return 0;      // the kernels index their threads with 32 bits: a zero grid fails loudly in check_launch
  long long g = (items + threads - 1) / threads;
  return (int)(g < 1 ? 1 : g);
}

// ------------------------------------------------------------------------------------------
// conv3x3, tiny Cin (<=4), NCHW input -> NHWC output.  One thread = one output pixel x 8 channels.
// Weights (f32 [9*Cin][Cout]) + bias staged in shared memory.
// ------------------------------------------------------------------------------------------
template <typename TI, typename TO>
__global__ void __launch_bounds__(256)
conv3x3_smallcin_kernel(const TI* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                        TO* __restrict__ y, int B, int Cin, int H, int W, int Cout, int Ho, int Wo, int stride,
                        int act) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sw[];  // [9*Cin*Cout] + [Cout]
  const int nw = 9 * Cin * Cout;
  for (int i = threadIdx.x; i < nw; i += blockDim.x) sw[i] = w[i];
  for (int i = threadIdx.x; i < Cout; i += blockDim.x) sw[nw + i] = bias ? bias[i] : 0.f;
  __syncthreads();
  const int groups = Cout >> 3;
  const long long total = (long long)B * Ho * Wo * groups;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(idx % groups);
    long long p = idx / groups;
    const int wo = (int)(p % Wo); p /= Wo;
    const int ho = (int)(p % Ho);
    const int b = (int)(p / Ho);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = sw[nw + g * 8 + j];
    const int hi0 = ho * stride - 1, wi0 = wo * stride - 1;
    for (int kh = 0; kh < 3; ++kh) {
      const int hi = hi0 + kh;
      if (hi < 0 || hi >= H) continue;
      for (int kw = 0; kw < 3; ++kw) {
        const int wi = wi0 + kw;
        if (wi < 0 || wi >= W) continue;
        for (int c = 0; c < Cin; ++c) {
          const float xv = to_f32<TI>(x[(((long long)b * Cin + c) * H + hi) * W + wi]);
          const float4* wp = reinterpret_cast<const float4*>(&sw[((kh * 3 + kw) * Cin + c) * Cout + g * 8]);
          const float4 w0 = wp[0], w1 = wp[1];
          acc[0] = fmaf(xv, w0.x, acc[0]); acc[1] = fmaf(xv, w0.y, acc[1]);
          acc[2] = fmaf(xv, w0.z, acc[2]); acc[3] = fmaf(xv, w0.w, acc[3]);
          acc[4] = fmaf(xv, w1.x, acc[4]); acc[5] = fmaf(xv, w1.y, acc[5]);
          acc[6] = fmaf(xv, w1.z, acc[6]); acc[7] = fmaf(xv, w1.w, acc[7]);
        }
      }
    }
    TO* yp = y + (((long long)b * Ho + ho) * Wo + wo) * Cout + g * 8;
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = apply_act_rt(acc[j], act);
    if (sizeof(TO) == 2) {
      uint4 t;
      t.x = pack_bf16x2(acc[0], acc[1]); t.y = pack_bf16x2(acc[2], acc[3]);
      t.z = pack_bf16x2(acc[4], acc[5]); t.w = pack_bf16x2(acc[6], acc[7]);
      *reinterpret_cast<uint4*>(yp) = t;
    } else {
      reinterpret_cast<float4*>(yp)[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
      reinterpret_cast<float4*>(yp)[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
  }
}


// ------------------------------------------------------------------------------------------
// conv3x3 Cin=3 on the tensor cores (bf16 output path).  K = 27 (padded to 32) is far too small for
// a TMA/tcgen05 pipeline and the NCHW planar, stride-2 input cannot be described by one TMA box, so
// the im2col fragment is gathered straight into registers and multiplied with warp-level
// mma.sync.m16n8k16 (bf16 x bf16 -> f32): a warp owns 16 consecutive output pixels x all Cout.
// Per pixel this needs ~1 load instruction + 0.5 MMA instead of 27 loads + 27 FMAs per 8 channels,
// which is what moves the kernel from issue-bound to HBM-bound.  k = c*9 + kh*3 + kw.
// Each CTA first stages the 3 channels x 3 input rows feeding 128 output pixels in shared memory with
// coalesced loads (every input element is read once per CTA), and the warps gather their fragments from
// there.  The C fragments are transposed through a per-warp shared-memory patch so that every thread
// stores whole 16-byte NHWC channel vectors (1 KB contiguous per warp).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <typename TI, int NT, int S>   // NT = Cout / 8, S = stride
__global__ void __launch_bounds__(256, NT <= 4 ? 4 : 2)
conv3x3_c3_mma_kernel(const TI* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                      __nv_bfloat16* __restrict__ y, int B, int H, int W, int Ho, int Wo, int act, int vec_ok) {
  pdl_trigger();
  pdl_wait();
  constexpr int Cout = NT * 8;
  constexpr int NCOL = 127 * S + 3;            // input columns feeding 128 output pixels
  constexpr int LEAD = 8;                      // the tile starts 8 columns left of the first output's centre so that
                                               // every 16-byte input vector is either fully inside or fully outside
  constexpr int JN = ((LEAD - 1 + NCOL) + 7) / 8 * 8;
  constexpr int PITCH = JN + 4;
  constexpr int VL = 16 / (int)sizeof(TI);     // elements per 16-byte global load
  __shared__ __align__(16) float tile[9][PITCH];   // [c*3 + kh][column]; column j <-> input column wo0*S - LEAD + j
  __shared__ __align__(16) __nv_bfloat16 patch[8][16][Cout + 8];   // +8: conflict-free fragment writes
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;

  // B fragments for both k-steps and all n-tiles: b0 = W[k=2t,2t+1][n=g], b1 = W[k=2t+8,2t+9][n=g]
  uint32_t bf[2][NT][2];
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int j = 0; j < NT; ++j)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int k = ks * 16 + h * 8 + 2 * t + e;          // k = c*9 + kh*3 + kw
          const int c = k / 9, r9 = k - c * 9;
          v[e] = (k < 27) ? __ldg(w + (r9 * 3 + c) * Cout + j * 8 + g) : 0.f;   // w is [kh][kw][c][Cout]
        }
        bf[ks][j][h] = pack_bf16x2(v[0], v[1]);
      }
  // this thread's 8 gather offsets into the smem tile (same for every pixel group): k -> (c*3+kh, kw)
  int koff[2][2][2];
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int k = ks * 16 + h * 8 + 2 * t + e;
        const int c = k / 9, r9 = k - c * 9;
        koff[ks][h][e] = (k < 27) ? (c * 3 + r9 / 3) * PITCH + r9 % 3 + (LEAD - 1) : -1;
      }
  float bias_v[NT][2];
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    bias_v[j][0] = bias ? __ldg(bias + j * 8 + 2 * t) : 0.f;
    bias_v[j][1] = bias ? __ldg(bias + j * 8 + 2 * t + 1) : 0.f;
  }

  const int segs = (Wo + 127) / 128;
  const long long total = (long long)B * Ho * segs;
  const long long HW = (long long)H * W;
  const float* tflat = &tile[0][0];
  for (long long job = blockIdx.x; job < total; job += gridDim.x) {
    const int sg = (int)(job % segs);
    long long p = job / segs;
    const int ho = (int)(p % Ho);
    const int b = (int)(p / Ho);
    const int wo0 = sg * 128;
    const TI* xb = x + (long long)b * 3 * HW;
    const int wi0 = wo0 * S - LEAD, hi0 = ho * S - 1;
    __syncthreads();                              // previous job's gathers are done
    if (vec_ok) {
      // 16-byte coalesced loads; W % VL == 0 and wi0 % VL == 0, so a vector never straddles the image border
      for (int i = threadIdx.x; i < 9 * (JN / VL); i += 256) {
        const int rowi = i / (JN / VL), v = i - rowi * (JN / VL);
        const int c = rowi / 3, kh = rowi - c * 3;
        const int hi = hi0 + kh, wi = wi0 + v * VL;
        float f[VL];
        if (hi >= 0 && hi < H && wi >= 0 && wi < W) {
          Vec16<TI> t;
          t.load(xb + (long long)c * HW + (long long)hi * W + wi);
#pragma unroll
          for (int e = 0; e < VL; ++e) f[e] = t.v[e];
        } else {
#pragma unroll
          for (int e = 0; e < VL; ++e) f[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < VL; e += 4)
          *reinterpret_cast<float4*>(&tile[rowi][v * VL + e]) = make_float4(f[e], f[e + 1], f[e + 2], f[e + 3]);
      }
    } else {
      for (int i = threadIdx.x; i < 9 * JN; i += 256) {
        const int rowi = i / JN, col = i - rowi * JN;
        const int c = rowi / 3, kh = rowi - c * 3;
        const int hi = hi0 + kh, wi = wi0 + col;
        float v = 0.f;
        if (hi >= 0 && hi < H && wi >= 0 && wi < W) v = to_f32<TI>(xb[(long long)c * HW + (long long)hi * W + wi]);
        tile[rowi][col] = v;
      }
    }
    __syncthreads();
    const int px0 = warp * 16;                    // this warp's 16 output pixels within the segment
    uint32_t afr[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int h = 0; h < 2; ++h)                 // h: k half (cols 2t.. / 2t+8..)
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {          // rr: row g / row g+8
          const int col = (px0 + g + rr * 8) * S;
          float v[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) v[e] = koff[ks][h][e] >= 0 ? tflat[koff[ks][h][e] + col] : 0.f;
          afr[ks][h * 2 + rr] = pack_bf16x2(v[0], v[1]);   // a0:(g,lo) a1:(g+8,lo) a2:(g,hi) a3:(g+8,hi)
        }
    float acc[NT][4];
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      acc[j][0] = bias_v[j][0]; acc[j][1] = bias_v[j][1]; acc[j][2] = bias_v[j][0]; acc[j][3] = bias_v[j][1];
    }
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int j = 0; j < NT; ++j) mma_bf16_16816(acc[j], afr[ks], bf[ks][j][0], bf[ks][j][1]);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      *reinterpret_cast<uint32_t*>(&patch[warp][g][j * 8 + 2 * t]) =
          pack_bf16x2(apply_act_rt(acc[j][0], act), apply_act_rt(acc[j][1], act));
      *reinterpret_cast<uint32_t*>(&patch[warp][g + 8][j * 8 + 2 * t]) =
          pack_bf16x2(apply_act_rt(acc[j][2], act), apply_act_rt(acc[j][3], act));
    }
    __syncwarp();
    __nv_bfloat16* yrow = y + (((long long)b * Ho + ho) * Wo + wo0 + px0) * Cout;
    for (int i = lane; i < 16 * NT; i += 32) {
      const int px = i / NT, cv = i - px * NT;
      if (wo0 + px0 + px < Wo)
        *reinterpret_cast<uint4*>(yrow + px * Cout + cv * 8) = *reinterpret_cast<const uint4*>(&patch[warp][px][cv * 8]);
    }
  }
}

// ------------------------------------------------------------------------------------------
// depthwise 3x3, NHWC.  One thread = TW consecutive output pixels along W x one 16-byte channel
// vector; the 3 x (TW-1)*S+3 input window is walked row by row so each input vector is loaded
// once per thread (sliding window in registers); neighbouring threads cover neighbouring channel
// vectors, so every load/store instruction of a warp is one contiguous run of 16-byte words.
// ------------------------------------------------------------------------------------------
template <typename T, int S, int TW>
__global__ void __launch_bounds__(256)
dwconv3x3_kernel(const T* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                 T* __restrict__ y, int B, int H, int W, int C, int Ho, int Wo, int act) {
  pdl_trigger();
  pdl_wait();
  using V = Vec16<T>;
  constexpr int VN = V::N;
  constexpr int NCOL = (TW - 1) * S + 3;
  const int cv = C / VN;
  const int strips = (Wo + TW - 1) / TW;
  const long long total = (long long)B * Ho * strips * cv;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  const int c0 = (int)(idx % (unsigned)cv) * VN;
  unsigned p = idx / (unsigned)cv;
  const int st = (int)(p % strips); p /= strips;
  const int ho = (int)(p % Ho);
  const int b = (int)(p / Ho);
  const int wo0 = st * TW;

  float acc[TW][VN];
  {
    float bv[VN];
#pragma unroll
    for (int j = 0; j < VN; ++j) bv[j] = bias ? __ldg(bias + c0 + j) : 0.f;
#pragma unroll
    for (int t = 0; t < TW; ++t)
#pragma unroll
      for (int j = 0; j < VN; ++j) acc[t][j] = bv[j];
  }
  const int wi0 = wo0 * S - 1;
#pragma unroll
  for (int kh = 0; kh < 3; ++kh) {
    const int hi = ho * S - 1 + kh;
    if (hi < 0 || hi >= H) continue;
    const T* row = x + (((long long)b * H + hi) * W) * C + c0;
    V in[NCOL];
#pragma unroll
    for (int i = 0; i < NCOL; ++i) {
      const int wi = wi0 + i;
      if (wi >= 0 && wi < W) {
        in[i].load(row + (long long)wi * C);
      } else {
#pragma unroll
        for (int j = 0; j < VN; ++j) in[i].v[j] = 0.f;
      }
    }
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      float wv[VN];
      const float* wp = w + (kh * 3 + kw) * C + c0;
#pragma unroll
      for (int j = 0; j < VN; j += 4) {
        const float4 t4 = __ldg(reinterpret_cast<const float4*>(wp + j));
        wv[j] = t4.x; wv[j + 1] = t4.y; wv[j + 2] = t4.z; wv[j + 3] = t4.w;
      }
#pragma unroll
      for (int t = 0; t < TW; ++t)
#pragma unroll
        for (int j = 0; j < VN; ++j) acc[t][j] = fmaf(in[t * S + kw].v[j], wv[j], acc[t][j]);
    }
  }
  T* yrow = y + (((long long)b * Ho + ho) * Wo) * C + c0;
#pragma unroll
  for (int t = 0; t < TW; ++t) {
    const int wo = wo0 + t;
    if (wo < Wo) {
      V o;
#pragma unroll
      for (int j = 0; j < VN; ++j) o.v[j] = apply_act_rt(acc[t][j], act);
      o.store(yrow + (long long)wo * C);
    }
  }
}

// ------------------------------------------------------------------------------------------
// depthwise 3x3, bf16 NHWC, 2-D register blocking: one thread = TH x TW output pixels x 8 channels.
// The (TH-1)*S+3 input rows are streamed one at a time: a row's (TW-1)*S+3 vectors are loaded with
// 16-byte loads, converted to f32 ONCE, and scattered into every output row/tap that uses them, so
// per output element the kernel issues ~4 loads/conversions instead of 9 and keeps only one input
// row live (registers -> occupancy).  fp32 accumulation, folded-BN shift + activation, bf16 store.
// ------------------------------------------------------------------------------------------
template <int S, int TW, int TH>
__global__ void __launch_bounds__(256, 2)
dwconv3x3_bf16_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                      __nv_bfloat16* __restrict__ y, int B, int H, int W, int C, int Ho, int Wo, int act) {
  pdl_trigger();
  pdl_wait();
  constexpr int NCOL = (TW - 1) * S + 3, NROW = (TH - 1) * S + 3;
  const int cv = C >> 3;
  const int sw_ = (Wo + TW - 1) / TW, sh_ = (Ho + TH - 1) / TH;
  const long long total = (long long)B * sh_ * sw_ * cv;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  const int c0 = (int)(idx % (unsigned)cv) << 3;
  unsigned p = idx / (unsigned)cv;
  const int tw = (int)(p % sw_); p /= sw_;
  const int th = (int)(p % sh_);
  const int b = (int)(p / sh_);
  const int wo0 = tw * TW, ho0 = th * TH;
  const int wi0 = wo0 * S - 1, hi0 = ho0 * S - 1;
  const float lo = act != B200SEG_ACT_NONE ? 0.f : -INFINITY, hi_ = act == B200SEG_ACT_RELU6 ? 6.f : INFINITY;

  float acc[TH][TW][8];
  {
    const float4 b0 = bias ? __ldg(reinterpret_cast<const float4*>(bias + c0)) : make_float4(0, 0, 0, 0);
    const float4 b1 = bias ? __ldg(reinterpret_cast<const float4*>(bias + c0 + 4)) : make_float4(0, 0, 0, 0);
#pragma unroll
    for (int o = 0; o < TH; ++o)
#pragma unroll
      for (int t = 0; t < TW; ++t) {
        acc[o][t][0] = b0.x; acc[o][t][1] = b0.y; acc[o][t][2] = b0.z; acc[o][t][3] = b0.w;
        acc[o][t][4] = b1.x; acc[o][t][5] = b1.y; acc[o][t][6] = b1.z; acc[o][t][7] = b1.w;
      }
  }
  const __nv_bfloat16* xb = x + (long long)b * H * W * C + c0;
#pragma unroll
  for (int r = 0; r < NROW; ++r) {
    const int hi = hi0 + r;
    if (hi < 0 || hi >= H) continue;            // zero padding row: contributes nothing
    const __nv_bfloat16* row = xb + (long long)hi * W * C;
    uint4 raw[NCOL];
#pragma unroll
    for (int i = 0; i < NCOL; ++i) {
      const int wi = wi0 + i;
      raw[i] = (wi >= 0 && wi < W) ? __ldg(reinterpret_cast<const uint4*>(row + (long long)wi * C)) : make_uint4(0, 0, 0, 0);
    }
    float in[NCOL][8];
#pragma unroll
    for (int i = 0; i < NCOL; ++i) {
      in[i][0] = bf16lo(raw[i].x); in[i][1] = bf16hi(raw[i].x); in[i][2] = bf16lo(raw[i].y); in[i][3] = bf16hi(raw[i].y);
      in[i][4] = bf16lo(raw[i].z); in[i][5] = bf16hi(raw[i].z); in[i][6] = bf16lo(raw[i].w); in[i][7] = bf16hi(raw[i].w);
    }
#pragma unroll
    for (int o = 0; o < TH; ++o) {
      const int kh = r - o * S;                 // compile-time after unrolling
      if (kh < 0 || kh > 2) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const float* wp = w + (kh * 3 + kw) * C + c0;
        const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp)), w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int t = 0; t < TW; ++t)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[o][t][j] = fmaf(in[t * S + kw][j], wv[j], acc[o][t][j]);
      }
    }
  }
#pragma unroll
  for (int o = 0; o < TH; ++o) {
    const int ho = ho0 + o;
    if (ho >= Ho) continue;
    __nv_bfloat16* yrow = y + (((long long)b * Ho + ho) * Wo) * C + c0;
#pragma unroll
    for (int t = 0; t < TW; ++t) {
      const int wo = wo0 + t;
      if (wo >= Wo) continue;
      float* a = acc[o][t];
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = fminf(fmaxf(a[j], lo), hi_);
      uint4 v;
      v.x = pack_bf16x2(a[0], a[1]); v.y = pack_bf16x2(a[2], a[3]);
      v.z = pack_bf16x2(a[4], a[5]); v.w = pack_bf16x2(a[6], a[7]);
      *reinterpret_cast<uint4*>(yrow + (long long)wo * C) = v;
    }
  }
}

// Same blocking with bf16 taps and the mixed-precision FMA (FHFMA.BF16: f32 += bf16 * bf16 from either register half):
// no unpack of the activations, the nine tap vectors of the thread's 8 channels stay in 36 registers for the whole tile.
// Arithmetic is identical to the f32-tap kernel for bf16-representable taps (products of two bf16 are exact in f32).
template <int S, int TW, int TH>
__global__ void __launch_bounds__(256, 2)
dwconv3x3_bf16w_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w, const float* __restrict__ bias,
                       __nv_bfloat16* __restrict__ y, int B, int H, int W, int C, int Ho, int Wo, int act) {
  pdl_trigger();
  pdl_wait();
  constexpr int NCOL = (TW - 1) * S + 3, NROW = (TH - 1) * S + 3;
  const int cv = C >> 3;
  const int sw_ = (Wo + TW - 1) / TW, sh_ = (Ho + TH - 1) / TH;
  const long long total = (long long)B * sh_ * sw_ * cv;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  const int c0 = (int)(idx % (unsigned)cv) << 3;
  unsigned p = idx / (unsigned)cv;
  const int tw = (int)(p % sw_); p /= sw_;
  const int th = (int)(p % sh_);
  const int b = (int)(p / sh_);
  const int wo0 = tw * TW, ho0 = th * TH;
  const int wi0 = wo0 * S - 1, hi0 = ho0 * S - 1;
  const float lo = act != B200SEG_ACT_NONE ? 0.f : -INFINITY, hi_ = act == B200SEG_ACT_RELU6 ? 6.f : INFINITY;

  uint4 wt[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) wt[k] = __ldg(reinterpret_cast<const uint4*>(w + (long long)k * C + c0));
  float acc[TH][TW][8];
  {
    const float4 b0 = bias ? __ldg(reinterpret_cast<const float4*>(bias + c0)) : make_float4(0, 0, 0, 0);
    const float4 b1 = bias ? __ldg(reinterpret_cast<const float4*>(bias + c0 + 4)) : make_float4(0, 0, 0, 0);
#pragma unroll
    for (int o = 0; o < TH; ++o)
#pragma unroll
      for (int t = 0; t < TW; ++t) {
        acc[o][t][0] = b0.x; acc[o][t][1] = b0.y; acc[o][t][2] = b0.z; acc[o][t][3] = b0.w;
        acc[o][t][4] = b1.x; acc[o][t][5] = b1.y; acc[o][t][6] = b1.z; acc[o][t][7] = b1.w;
      }
  }
  const __nv_bfloat16* xb = x + (long long)b * H * W * C + c0;
#pragma unroll
  for (int r = 0; r < NROW; ++r) {
    const int hi = hi0 + r;
    if (hi < 0 || hi >= H) continue;            // zero padding row: contributes nothing
    const __nv_bfloat16* row = xb + (long long)hi * W * C;
    uint4 raw[NCOL];
#pragma unroll
    for (int i = 0; i < NCOL; ++i) {
      const int wi = wi0 + i;
      raw[i] = (wi >= 0 && wi < W) ? __ldg(reinterpret_cast<const uint4*>(row + (long long)wi * C)) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int o = 0; o < TH; ++o) {
      const int kh = r - o * S;                 // compile-time after unrolling
      if (kh < 0 || kh > 2) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const uint4 wv = wt[kh * 3 + kw];
#pragma unroll
        for (int t = 0; t < TW; ++t) {
          const uint4 xv = raw[t * S + kw];
          float* a = acc[o][t];
          a[0] = fma_bf16_lo(xv.x, wv.x, a[0]); a[1] = fma_bf16_hi(xv.x, wv.x, a[1]);
          a[2] = fma_bf16_lo(xv.y, wv.y, a[2]); a[3] = fma_bf16_hi(xv.y, wv.y, a[3]);
          a[4] = fma_bf16_lo(xv.z, wv.z, a[4]); a[5] = fma_bf16_hi(xv.z, wv.z, a[5]);
          a[6] = fma_bf16_lo(xv.w, wv.w, a[6]); a[7] = fma_bf16_hi(xv.w, wv.w, a[7]);
        }
      }
    }
  }
#pragma unroll
  for (int o = 0; o < TH; ++o) {
    const int ho = ho0 + o;
    if (ho >= Ho) continue;
    __nv_bfloat16* yrow = y + (((long long)b * Ho + ho) * Wo) * C + c0;
#pragma unroll
    for (int t = 0; t < TW; ++t) {
      const int wo = wo0 + t;
      if (wo >= Wo) continue;
      float* a = acc[o][t];
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = fminf(fmaxf(a[j], lo), hi_);
      uint4 v;
      v.x = pack_bf16x2(a[0], a[1]); v.y = pack_bf16x2(a[2], a[3]);
      v.z = pack_bf16x2(a[4], a[5]); v.w = pack_bf16x2(a[6], a[7]);
      *reinterpret_cast<uint4*>(yrow + (long long)wo * C) = v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// y[b,ho,wo,0:Cs] = skip ; y[b,ho,wo,Cs:] = bilinear x2 (align_corners=False) of x.
// One thread = one 16-byte channel vector of a 2x2 block of output pixels: the 3x3 source
// neighbourhood is loaded and converted once (9 loads for 4 outputs instead of 16) and the
// interpolation is done separably -- for scale 2 the weights are exactly {0.25, 0.75}; clamped
// neighbour indices reproduce PyTorch's border rule (src = max(0, (dst+0.5)/2 - 0.5)) because
// 0.25*a + 0.75*a == a exactly in one fma.
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
upsample2x_concat_kernel(const T* __restrict__ skip, const T* __restrict__ x, T* __restrict__ y, int B, int h,
                         int w, int Cs, int Cu) {
  pdl_trigger();
  pdl_wait();
  using V = Vec16<T>;
  constexpr int VN = V::N;
  const int C = Cs + Cu, cvs = Cs / VN, cvu = Cu / VN, Wo = 2 * w;
  // When the skip slice ends on a 32-byte sector boundary, threads [0, n_skip) copy the skip slice and the rest interpolate:
  // warps are uniform (with the two kinds interleaved along the channel axis every warp of the 48-channel stage executed
  // both paths).  Otherwise (24 skip channels: 48 bytes) the two kinds stay interleaved so that the sector shared by the
  // two slices of a pixel is written by neighbouring lanes at the same time (split, that stage was 30 % slower).
  const unsigned npix = (unsigned)B * h * w, total = npix * (cvs + cvu);
  unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  int c;
  unsigned p;
  if ((Cs * (int)sizeof(T)) % 32 == 0) {
    const unsigned n_skip = npix * cvs;
    const bool is_skip = idx < n_skip;
    if (!is_skip) idx -= n_skip;
    const unsigned cv = is_skip ? cvs : cvu;
    c = (int)(idx % cv) * VN + (is_skip ? 0 : Cs);
    p = idx / cv;
  } else {
    const unsigned cv = cvs + cvu;
    c = (int)(idx % cv) * VN;
    p = idx / cv;
  }
  const int j = (int)(p % w); p /= w;
  const int i = (int)(p % h);
  const int b = (int)(p / h);
  T* y00 = y + (((long long)b * 2 * h + 2 * i) * Wo + 2 * j) * C + c;     // output pixel (2i, 2j)
  const long long yrow = (long long)Wo * C;
  if (c < Cs) {
    const T* s00 = skip + (((long long)b * 2 * h + 2 * i) * Wo + 2 * j) * Cs + c;
    const long long srow = (long long)Wo * Cs;
    const uint4 a0 = __ldg(reinterpret_cast<const uint4*>(s00)), a1 = __ldg(reinterpret_cast<const uint4*>(s00 + Cs));
    const uint4 a2 = __ldg(reinterpret_cast<const uint4*>(s00 + srow)), a3 = __ldg(reinterpret_cast<const uint4*>(s00 + srow + Cs));
    *reinterpret_cast<uint4*>(y00) = a0; *reinterpret_cast<uint4*>(y00 + C) = a1;
    *reinterpret_cast<uint4*>(y00 + yrow) = a2; *reinterpret_cast<uint4*>(y00 + yrow + C) = a3;
    return;
  }
  const int cu = c - Cs;
  const int ri[3] = {max(i - 1, 0), i, min(i + 1, h - 1)};
  const int qj[3] = {max(j - 1, 0), j, min(j + 1, w - 1)};
  const T* xb = x + (long long)b * h * w * Cu + cu;
  float te[3][VN], to[3][VN];     // vertically blended columns for the even / odd output row
  if constexpr (sizeof(T) == 2) {
    // bf16: the same arithmetic on the packed vectors as loaded, through the mixed-precision FMA (f32 = bf16 * bf16 + f32;
    // 0.25 and 0.75 are bf16 numbers, the products are exact): no unpack instructions.  All nine loads are issued before
    // the first FMA: a run-time-zero word derived from every loaded vector is OR-ed into the two weight constants (ptxas
    // otherwise sinks the loads into the arithmetic, three in flight per thread).
    uint4 a[3], m[3], d[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      a[q] = __ldg(reinterpret_cast<const uint4*>(xb + ((long long)ri[0] * w + qj[q]) * Cu));
      m[q] = __ldg(reinterpret_cast<const uint4*>(xb + ((long long)ri[1] * w + qj[q]) * Cu));
      d[q] = __ldg(reinterpret_cast<const uint4*>(xb + ((long long)ri[2] * w + qj[q]) * Cu));
    }
    uint32_t dep = 0;
#pragma unroll
    for (int q = 0; q < 3; ++q) dep |= a[q].x | m[q].x | d[q].x;
    dep &= (uint32_t)B >> 30;                                        // B < 2^30: zero, but not provably so
    const uint32_t Q25 = 0x3E803E80u | dep, Q75 = 0x3F403F40u | dep;   // bf16x2 {0.25, 0.25}, {0.75, 0.75}
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const uint32_t av[4] = {a[q].x, a[q].y, a[q].z, a[q].w}, mv[4] = {m[q].x, m[q].y, m[q].z, m[q].w},
                     dv[4] = {d[q].x, d[q].y, d[q].z, d[q].w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        te[q][2 * k] = fma_bf16_lo(mv[k], Q75, fma_bf16_lo(av[k], Q25, 0.f));
        te[q][2 * k + 1] = fma_bf16_hi(mv[k], Q75, fma_bf16_hi(av[k], Q25, 0.f));
        to[q][2 * k] = fma_bf16_lo(mv[k], Q75, fma_bf16_lo(dv[k], Q25, 0.f));
        to[q][2 * k + 1] = fma_bf16_hi(mv[k], Q75, fma_bf16_hi(dv[k], Q25, 0.f));
      }
    }
  } else {
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      V a, m, d;
      a.load(xb + ((long long)ri[0] * w + qj[q]) * Cu);
      m.load(xb + ((long long)ri[1] * w + qj[q]) * Cu);
      d.load(xb + ((long long)ri[2] * w + qj[q]) * Cu);
#pragma unroll
      for (int k = 0; k < VN; ++k) {
        te[q][k] = fmaf(m.v[k], 0.75f, 0.25f * a.v[k]);
        to[q][k] = fmaf(m.v[k], 0.75f, 0.25f * d.v[k]);
      }
    }
  }
  V o;
#pragma unroll
  for (int k = 0; k < VN; ++k) o.v[k] = fmaf(te[1][k], 0.75f, 0.25f * te[0][k]);
  o.store(y00);
#pragma unroll
  for (int k = 0; k < VN; ++k) o.v[k] = fmaf(te[1][k], 0.75f, 0.25f * te[2][k]);
  o.store(y00 + C);
#pragma unroll
  for (int k = 0; k < VN; ++k) o.v[k] = fmaf(to[1][k], 0.75f, 0.25f * to[0][k]);
  o.store(y00 + yrow);
#pragma unroll
  for (int k = 0; k < VN; ++k) o.v[k] = fmaf(to[1][k], 0.75f, 0.25f * to[2][k]);
  o.store(y00 + yrow + C);
}

// ------------------------------------------------------------------------------------------
// The upsample alone (Cs = 0, bf16): what the decoder's two-source convolutions read next to the skip tensor.
// One thread = one 16-byte channel vector of a 2 x 2KW block of output pixels: the source window of 3 rows x (KW + 2)
// columns is loaded once and slid along the row, so the low-resolution input is read 3(KW+2)/KW times per output
// vector pair instead of 9/1 (2x fewer load instructions and L1 traffic for KW = 4), and each thread issues 4KW
// independent 16-byte stores.  Same arithmetic in the same order as upsample2x_concat_kernel (bit-identical).
// ------------------------------------------------------------------------------------------
template <int KW>
__global__ void __launch_bounds__(256)
upsample2x_bf16_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y, int B, int h, int w, int Cu) {
  pdl_trigger();
  pdl_wait();
  const int cv = Cu / 8, wg = (w + KW - 1) / KW, Wo = 2 * w;
  const unsigned total = (unsigned)B * h * wg * cv;
  unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher)
  if (idx >= total) return;
  const int c = (int)(idx % cv) * 8;
  unsigned p = idx / cv;
  const int j0 = (int)(p % wg) * KW; p /= wg;
  const int i = (int)(p % h);
  const int b = (int)(p / h);
  const __nv_bfloat16* xb = x + (long long)b * h * w * Cu + c;
  const long long r0 = (long long)max(i - 1, 0) * w, r1 = (long long)i * w, r2 = (long long)min(i + 1, h - 1) * w;
  uint4 a[KW + 2], m[KW + 2], d[KW + 2];     // source columns j0-1 .. j0+KW (clamped) of rows i-1, i, i+1
#pragma unroll
  for (int q = 0; q < KW + 2; ++q) {
    const int jq = min(max(j0 + q - 1, 0), w - 1);
    a[q] = Vec16<__nv_bfloat16>::ldraw(xb + (r0 + jq) * Cu);
    m[q] = Vec16<__nv_bfloat16>::ldraw(xb + (r1 + jq) * Cu);
    d[q] = Vec16<__nv_bfloat16>::ldraw(xb + (r2 + jq) * Cu);
  }
  const uint32_t Q25 = 0x3E803E80u, Q75 = 0x3F403F40u;     // bf16x2 {0.25, 0.25}, {0.75, 0.75}
  float te[KW + 2][8], to[KW + 2][8];       // vertically blended columns for the even / odd output row
#pragma unroll
  for (int q = 0; q < KW + 2; ++q) {
    const uint32_t av[4] = {a[q].x, a[q].y, a[q].z, a[q].w}, mv[4] = {m[q].x, m[q].y, m[q].z, m[q].w},
                   dv[4] = {d[q].x, d[q].y, d[q].z, d[q].w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      te[q][2 * k] = fma_bf16_lo(mv[k], Q75, fma_bf16_lo(av[k], Q25, 0.f));
      te[q][2 * k + 1] = fma_bf16_hi(mv[k], Q75, fma_bf16_hi(av[k], Q25, 0.f));
      to[q][2 * k] = fma_bf16_lo(mv[k], Q75, fma_bf16_lo(dv[k], Q25, 0.f));
      to[q][2 * k + 1] = fma_bf16_hi(mv[k], Q75, fma_bf16_hi(dv[k], Q25, 0.f));
    }
  }
  __nv_bfloat16* y0 = y + (((long long)b * 2 * h + 2 * i) * Wo + 2 * j0) * Cu + c;     // output pixel (2i, 2j0)
  const long long yrow = (long long)Wo * Cu;
#pragma unroll
  for (int t = 0; t < KW; ++t) {
    if (j0 + t >= w) break;
    __nv_bfloat16* yp = y0 + (long long)(2 * t) * Cu;
    Vec16<__nv_bfloat16> o;
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = fmaf(te[t + 1][k], 0.75f, 0.25f * te[t][k]);
    o.store(yp);
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = fmaf(te[t + 1][k], 0.75f, 0.25f * te[t + 2][k]);
    o.store(yp + Cu);
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = fmaf(to[t + 1][k], 0.75f, 0.25f * to[t][k]);
    o.store(yp + yrow);
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = fmaf(to[t + 1][k], 0.75f, 0.25f * to[t + 2][k]);
    o.store(yp + yrow + Cu);
  }
}

// 16 channels of one NHWC pixel as floats (ldc == 16: 32 B bf16 / 64 B f32, 16-byte vector loads)
template <typename T>
__device__ __forceinline__ void load_px16(const T* p, float (&v)[16]);
template <>
__device__ __forceinline__ void load_px16<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[16]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p) + 1);
  v[0] = bf16lo(a.x); v[1] = bf16hi(a.x); v[2] = bf16lo(a.y); v[3] = bf16hi(a.y);
  v[4] = bf16lo(a.z); v[5] = bf16hi(a.z); v[6] = bf16lo(a.w); v[7] = bf16hi(a.w);
  v[8] = bf16lo(b.x); v[9] = bf16hi(b.x); v[10] = bf16lo(b.y); v[11] = bf16hi(b.y);
  v[12] = bf16lo(b.z); v[13] = bf16hi(b.z); v[14] = bf16lo(b.w); v[15] = bf16hi(b.w);
}
template <>
__device__ __forceinline__ void load_px16<float>(const float* p, float (&v)[16]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p) + i);
    v[4 * i] = a.x; v[4 * i + 1] = a.y; v[4 * i + 2] = a.z; v[4 * i + 3] = a.w;
  }
}

// One thread = PPT consecutive output pixels along W of one output row.  The two source rows are
// fixed per thread, so each source column is first blended vertically (hy*row0 + ly*row1) when it is
// loaded; consecutive outputs advance the source column by < 0.5, so the thread walks its source
// columns with a two-column register window and loads every logits pixel once, with 16-byte loads.
// Stores are contiguous along W per class plane (8/16-byte vectors).
template <typename T, typename TO, int PPT, int CMAX, bool ARGMAX>
__global__ void __launch_bounds__(256, 3)      // 80 registers: 3 blocks/SM measured 99 us vs 115 (2 blocks) and 113 (4, spills)
upsample2x_ac_kernel(const T* __restrict__ lg, TO* __restrict__ out, uint8_t* __restrict__ mask, int B, int h, int w,
                     int C) {
  pdl_trigger();
  pdl_wait();
  const int Ho = 2 * h, Wo = 2 * w;
  const int wq = Wo / PPT;
  const long long total = (long long)B * Ho * wq;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  const int q = (int)(idx % (unsigned)wq);
  unsigned p = idx / (unsigned)wq;
  const int ho = (int)(p % Ho);
  const int b = (int)(p / Ho);
  const float sch = (Ho > 1) ? (float)(h - 1) / (float)(Ho - 1) : 0.f;
  const float scw = (Wo > 1) ? (float)(w - 1) / (float)(Wo - 1) : 0.f;
  const float sy = sch * ho;
  const int y0 = (int)sy;
  const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
  const float ly = sy - y0, hy = 1.f - ly;
  const T* r0 = lg + ((long long)b * h + y0) * w * 16;
  const T* r1 = lg + ((long long)b * h + y1) * w * 16;

  auto load_col = [&](int xcol, float (&dst)[CMAX]) {
    float a[16], c[16];
    load_px16<T>(r0 + (long long)xcol * 16, a);
    load_px16<T>(r1 + (long long)xcol * 16, c);
#pragma unroll
    for (int i = 0; i < CMAX; ++i) dst[i] = hy * a[i] + ly * c[i];
  };
  int xc = (int)(scw * (q * PPT));
  float lft[CMAX], rgt[CMAX];
  load_col(xc, lft);
  load_col(xc + (xc < w - 1 ? 1 : 0), rgt);
  float res[PPT][CMAX];
#pragma unroll
  for (int t = 0; t < PPT; ++t) {
    const int wo = q * PPT + t;
    const float sx = scw * wo;
    const int x0 = (int)sx;
    if (x0 != xc) {   // advance the window by one column
      xc = x0;
#pragma unroll
      for (int i = 0; i < CMAX; ++i) lft[i] = rgt[i];
      load_col(xc + (xc < w - 1 ? 1 : 0), rgt);
    }
    const float lx = sx - x0, hx = 1.f - lx;
#pragma unroll
    for (int i = 0; i < CMAX; ++i) res[t][i] = hx * lft[i] + lx * rgt[i];
  }
  if (ARGMAX) {
    uint32_t packed = 0;
#pragma unroll
    for (int t = 0; t < PPT; ++t) {
      int best = 0;
      float bv = res[t][0];
#pragma unroll
      for (int c = 1; c < CMAX; ++c)
        if (c < C && res[t][c] > bv) { bv = res[t][c]; best = c; }   // first max wins, like torch.max
      packed |= (uint32_t)best << (8 * t);
    }
    static_assert(!ARGMAX || PPT == 4, "argmax variant packs 4 pixels per 32-bit store");
    *reinterpret_cast<uint32_t*>(mask + ((long long)b * Ho + ho) * Wo + q * PPT) = packed;
  } else {
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < C) {
        TO* op = out + (((long long)b * C + c) * Ho + ho) * Wo + q * PPT;
        if (sizeof(TO) == 2 && PPT == 4) {
          uint2 v;
          v.x = pack_bf16x2(res[0][c], res[1][c]); v.y = pack_bf16x2(res[2][c], res[3][c]);
          *reinterpret_cast<uint2*>(op) = v;
        } else if (sizeof(TO) == 4 && PPT == 4) {
          *reinterpret_cast<float4*>(op) = make_float4(res[0][c], res[1][c], res[2][c], res[3][c]);
        } else {
#pragma unroll
          for (int t = 0; t < PPT; ++t) op[t] = from_f32<TO>(res[t][c]);
        }
      }
    }
  }
}

template <typename T, typename TO>
__global__ void __launch_bounds__(256)
nhwc_to_nchw_kernel(const T* __restrict__ x, int ldc, TO* __restrict__ out, int B, int H, int W, int C) {
  pdl_trigger();
  pdl_wait();
  const long long total = (long long)B * H * W;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  const unsigned hw = (unsigned)H * W;
  const int b = (int)(idx / hw);
  const long long pix = idx % hw;
  const T* xp = x + (long long)idx * ldc;
  for (int c = 0; c < C; ++c) out[((long long)b * C + c) * hw + pix] = from_f32<TO>(to_f32<T>(xp[c]));
}

template <typename T>
__global__ void __launch_bounds__(256)
maxpool2x2_kernel(const T* __restrict__ x, T* __restrict__ y, int B, int H, int W, int C) {
  pdl_trigger();
  pdl_wait();
  using V = Vec16<T>;
  constexpr int VN = V::N;
  const int Ho = H / 2, Wo = W / 2, cv = C / VN;
  const long long total = (long long)B * Ho * Wo * cv;
  const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^31 threads (checked by the launcher): 32-bit div/mod
  if (idx >= total) return;
  const int c = (int)(idx % (unsigned)cv) * VN;
  unsigned p = idx / (unsigned)cv;
  const int wo = (int)(p % Wo); p /= Wo;
  const int ho = (int)(p % Ho);
  const int b = (int)(p / Ho);
  const T* xp = x + (((long long)b * H + 2 * ho) * W + 2 * wo) * C + c;
  V a, bq, cq, d, o;
  a.load(xp); bq.load(xp + C); cq.load(xp + (long long)W * C); d.load(xp + (long long)W * C + C);
#pragma unroll
  for (int j = 0; j < VN; ++j) o.v[j] = fmaxf(fmaxf(a.v[j], bq.v[j]), fmaxf(cq.v[j], d.v[j]));
  o.store(y + (((long long)b * Ho + ho) * Wo + wo) * C + c);
}

}  // namespace b200

using namespace b200;
typedef __nv_bfloat16 bf16;

extern "C" {

int b200seg_conv3x3_smallcin(const void* x, int x_dtype, const float* w, const float* b, void* y, int y_dtype,
                             int B, int Cin, int H, int W, int Cout, int stride, int act, b200seg_stream_t s) {
  B200_REQUIRE(Cin >= 1 && Cin <= 4, "conv3x3_smallcin: Cin=%d not in 1..4", Cin);
  B200_REQUIRE(Cout % 8 == 0 && Cout <= 256, "conv3x3_smallcin: Cout=%d must be a multiple of 8, <=256", Cout);
  B200_REQUIRE(stride == 1 || stride == 2, "conv3x3_smallcin: stride=%d", stride);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "conv3x3_smallcin: empty tensor");
  const int Ho = (H + 2 - 3) / stride + 1, Wo = (W + 2 - 3) / stride + 1;
  const long long total = (long long)B * Ho * Wo * (Cout / 8);
  const int threads = 256;
  long long g = (total + threads - 1) / threads;
  const long long cap = (long long)sm_count() * 8;
  if (g > cap) g = cap;   // grid-stride: amortise the weight staging
  const size_t smem = (size_t)(9 * Cin * Cout + Cout) * sizeof(float);
  cudaStream_t st = (cudaStream_t)s;
  if (y_dtype == B200SEG_BF16 && Cin == 3 && (Cout == 32 || Cout == 64 || Cout == 16)) {
    // tensor-core path (bf16 storage): one warp = 16 output pixels x all Cout
    const long long jobs = (long long)B * Ho * ((Wo + 127) / 128);
    long long gb = jobs;
    const long long capb = (long long)sm_count() * 8;
    if (gb > capb) gb = capb;
#define LAUNCH_MMA(TI, NT)                                                                                              \
  {                                                                                                                     \
    const int vl = 16 / (int)sizeof(TI);                                                                                \
    const int vok = (W % vl == 0) && (((uintptr_t)x & 15) == 0);                                                        \
    if (stride == 2) launch_pdl(conv3x3_c3_mma_kernel<TI, NT, 2>, dim3((unsigned)(int)gb), dim3((unsigned)256), (size_t)0, st, (const TI*)x, w, b, (bf16*)y, B, H, W, Ho, Wo, act, vok); \
    else launch_pdl(conv3x3_c3_mma_kernel<TI, NT, 1>, dim3((unsigned)(int)gb), dim3((unsigned)256), (size_t)0, st, (const TI*)x, w, b, (bf16*)y, B, H, W, Ho, Wo, act, vok);             \
  }
    if (x_dtype == B200SEG_F32) { if (Cout == 32) LAUNCH_MMA(float, 4) else if (Cout == 64) LAUNCH_MMA(float, 8) else LAUNCH_MMA(float, 2) }
    else if (x_dtype == B200SEG_BF16) { if (Cout == 32) LAUNCH_MMA(bf16, 4) else if (Cout == 64) LAUNCH_MMA(bf16, 8) else LAUNCH_MMA(bf16, 2) }
    else return set_error(-1, "conv3x3_smallcin: bad x dtype %d", x_dtype);
#undef LAUNCH_MMA
    return check_launch("conv3x3_c3_mma");
  }
#define LAUNCH(TI, TO)                                                                                      \
  launch_pdl(conv3x3_smallcin_kernel<TI, TO>, dim3((unsigned)(int)g), dim3((unsigned)threads), (size_t)smem, st, (const TI*)x, w, b, (TO*)y, B, Cin, H, W, \
                                                                 Cout, Ho, Wo, stride, act)
  if (x_dtype == B200SEG_F32 && y_dtype == B200SEG_F32) LAUNCH(float, float);
  else if (x_dtype == B200SEG_F32 && y_dtype == B200SEG_BF16) LAUNCH(float, bf16);
  else if (x_dtype == B200SEG_BF16 && y_dtype == B200SEG_BF16) LAUNCH(bf16, bf16);
  else if (x_dtype == B200SEG_BF16 && y_dtype == B200SEG_F32) LAUNCH(bf16, float);
  else return set_error(-1, "conv3x3_smallcin: bad dtypes %d %d", x_dtype, y_dtype);
#undef LAUNCH
  return check_launch("conv3x3_smallcin");
}

int b200seg_dwconv3x3(const void* x, const float* w, const float* b, void* y, int dtype, int B, int H, int W,
                      int C, int stride, int act, b200seg_stream_t s) {
  const int vn = dtype == B200SEG_BF16 ? 8 : 4;
  B200_REQUIRE(dtype == B200SEG_BF16 || dtype == B200SEG_F32, "dwconv3x3: bad dtype %d", dtype);
  B200_REQUIRE(C % vn == 0, "dwconv3x3: C=%d must be a multiple of %d", C, vn);
  B200_REQUIRE(stride == 1 || stride == 2, "dwconv3x3: stride=%d", stride);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "dwconv3x3: empty tensor");
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  cudaStream_t st = (cudaStream_t)s;
  const int threads = 256;
#define LAUNCH(T, S, TW)                                                                              \
  {                                                                                                   \
    const long long total = (long long)B * Ho * ((Wo + TW - 1) / TW) * (C / vn);                       \
    launch_pdl(dwconv3x3_kernel<T, S, TW>, dim3((unsigned)grid_for(total, threads)), dim3((unsigned)threads), (size_t)0, st, (const T*)x, w, b, (T*)y, \
                                                                             B, H, W, C, Ho, Wo, act); \
  }
  if (dtype == B200SEG_BF16) {
    static int variant = -1;      // tuning knob (B200SEG_DW_VARIANT): 0 = default
    if (variant < 0) { const char* e = getenv("B200SEG_DW_VARIANT"); variant = e ? atoi(e) : 0; }
#define LAUNCH2(S, TW, TH)                                                                                        \
  {                                                                                                               \
    const long long total = (long long)B * ((Ho + TH - 1) / TH) * ((Wo + TW - 1) / TW) * (C / 8);                 \
    launch_pdl(dwconv3x3_bf16_kernel<S, TW, TH>, dim3((unsigned)grid_for(total, threads)), dim3((unsigned)threads), (size_t)0, st, (const bf16*)x, w, b, (bf16*)y, \
                                                                                   B, H, W, C, Ho, Wo, act);      \
  }
    if (stride == 1) {
      if (variant == 1) LAUNCH2(1, 2, 1) else if (variant == 2) LAUNCH2(1, 4, 1) else if (variant == 3) LAUNCH2(1, 4, 2)
      else if (variant == 9) LAUNCH(bf16, 1, 4) else if (variant == 4) LAUNCH2(1, 2, 2) else LAUNCH2(1, 4, 2)   // default: 4x2 block (measured best)
    } else {
      if (variant == 1) LAUNCH2(2, 2, 1) else if (variant == 2) LAUNCH2(2, 4, 1) else if (variant == 3) LAUNCH2(2, 1, 2)
      else if (variant == 9) LAUNCH(bf16, 2, 2) else if (variant == 4) LAUNCH2(2, 2, 2) else LAUNCH2(2, 4, 1)   // default: 4x1 strip (measured best)
    }
#undef LAUNCH2
  } else {
    if (stride == 1) LAUNCH(float, 1, 4) else LAUNCH(float, 2, 2)
  }
#undef LAUNCH
  return check_launch("dwconv3x3");
}

int b200seg_dwconv3x3_bf16w(const void* x, const void* w, const float* b, void* y, int B, int H, int W, int C, int stride,
                            int act, int variant, b200seg_stream_t s) {
  B200_REQUIRE(C > 0 && C % 8 == 0, "dwconv3x3_bf16w: C=%d must be a positive multiple of 8", C);
  B200_REQUIRE(stride == 1 || stride == 2, "dwconv3x3_bf16w: stride=%d", stride);
  B200_REQUIRE(B > 0 && H > 0 && W > 0 && x && w && y, "dwconv3x3_bf16w: bad arguments");
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  cudaStream_t st = (cudaStream_t)s;
  const int threads = 256;
#define LAUNCHW(S, TW, TH)                                                                                        \
  {                                                                                                               \
    const long long total = (long long)B * ((Ho + TH - 1) / TH) * ((Wo + TW - 1) / TW) * (C / 8);                 \
    launch_pdl(dwconv3x3_bf16w_kernel<S, TW, TH>, dim3((unsigned)grid_for(total, threads)), dim3((unsigned)threads), (size_t)0, st, (const bf16*)x, (const bf16*)w, b, (bf16*)y, \
               B, H, W, C, Ho, Wo, act);                                                                          \
  }
  if (stride == 1) {
    if (variant == 1) LAUNCHW(1, 4, 1) else if (variant == 2) LAUNCHW(1, 2, 2) else if (variant == 3) LAUNCHW(1, 4, 4) else LAUNCHW(1, 4, 2)
  } else {
    if (variant == 1) LAUNCHW(2, 2, 1) else if (variant == 2) LAUNCHW(2, 2, 2) else if (variant == 3) LAUNCHW(2, 4, 2) else LAUNCHW(2, 4, 1)
  }
#undef LAUNCHW
  return check_launch("dwconv3x3_bf16w");
}

int b200seg_upsample2x_concat(const void* skip, const void* x, void* y, int dtype, int B, int h, int w, int Cs,
                              int Cu, b200seg_stream_t s) {
  const int vn = dtype == B200SEG_BF16 ? 8 : 4;
  B200_REQUIRE(dtype == B200SEG_BF16 || dtype == B200SEG_F32, "upsample2x_concat: bad dtype %d", dtype);
  B200_REQUIRE(Cs % vn == 0 && Cu % vn == 0 && Cu > 0 && Cs >= 0, "upsample2x_concat: Cs=%d Cu=%d must be multiples of %d", Cs, Cu, vn);
  B200_REQUIRE(B > 0 && h > 0 && w > 0, "upsample2x_concat: empty tensor");
  const long long total = (long long)B * h * w * ((Cs + Cu) / vn);     // one thread per 2x2 output block x vector
  cudaStream_t st = (cudaStream_t)s;
  if (dtype == B200SEG_BF16 && Cs == 0) {
    constexpr int KW = 4;
    const long long n = (long long)B * h * ((w + KW - 1) / KW) * (Cu / vn);
    launch_pdl(upsample2x_bf16_kernel<KW>, dim3((unsigned)grid_for(n, 256)), dim3((unsigned)256), (size_t)0, st, (const bf16*)x, (bf16*)y, B, h, w, Cu);
  } else if (dtype == B200SEG_BF16)
    launch_pdl(upsample2x_concat_kernel<bf16>, dim3((unsigned)grid_for(total, 256)), dim3((unsigned)256), (size_t)0, st, (const bf16*)skip, (const bf16*)x, (bf16*)y, B, h, w, Cs, Cu);
  else
    launch_pdl(upsample2x_concat_kernel<float>, dim3((unsigned)grid_for(total, 256)), dim3((unsigned)256), (size_t)0, st, (const float*)skip, (const float*)x, (float*)y, B, h, w, Cs, Cu);
  return check_launch("upsample2x_concat");
}

int b200seg_upsample2x_ac_nchw(const void* logits, int dtype, int ldc, void* out, int out_dtype, int B, int h,
                               int w, int C, b200seg_stream_t s) {
  B200_REQUIRE(C >= 1 && C <= 16 && ldc == 16, "upsample2x_ac_nchw: C=%d (<=16), ldc=%d (must be 16)", C, ldc);
  B200_REQUIRE(B > 0 && h > 0 && w > 0, "upsample2x_ac_nchw: empty tensor");
  cudaStream_t st = (cudaStream_t)s;
  const bool v4 = (2 * w) % 4 == 0;
  const long long total = (long long)B * 2 * h * (2 * w / (v4 ? 4 : 2));
  const int g = grid_for(total, 256);
#define LAUNCH(T, TO)                                                                                               \
  {                                                                                                                 \
    if (v4 && C <= 12) launch_pdl(upsample2x_ac_kernel<T, TO, 4, 12, false>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const T*)logits, (TO*)out, nullptr, B, h, w, C); \
    else if (v4) launch_pdl(upsample2x_ac_kernel<T, TO, 4, 16, false>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const T*)logits, (TO*)out, nullptr, B, h, w, C);       \
    else launch_pdl(upsample2x_ac_kernel<T, TO, 2, 16, false>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const T*)logits, (TO*)out, nullptr, B, h, w, C);               \
  }
  if (dtype == B200SEG_BF16 && out_dtype == B200SEG_BF16) LAUNCH(bf16, bf16)
  else if (dtype == B200SEG_BF16 && out_dtype == B200SEG_F32) LAUNCH(bf16, float)
  else if (dtype == B200SEG_F32 && out_dtype == B200SEG_F32) LAUNCH(float, float)
  else if (dtype == B200SEG_F32 && out_dtype == B200SEG_BF16) LAUNCH(float, bf16)
  else return set_error(-1, "upsample2x_ac_nchw: bad dtypes");
#undef LAUNCH
  return check_launch("upsample2x_ac_nchw");
}

int b200seg_upsample2x_ac_argmax(const void* logits, int dtype, int ldc, uint8_t* mask, int B, int h, int w, int C,
                                 b200seg_stream_t s) {
  B200_REQUIRE(C >= 1 && C <= 16 && ldc == 16, "upsample2x_ac_argmax: C=%d (<=16), ldc=%d (must be 16)", C, ldc);
  B200_REQUIRE(B > 0 && h > 0 && w > 0 && (2 * w) % 4 == 0, "upsample2x_ac_argmax: bad shape");
  cudaStream_t st = (cudaStream_t)s;
  const long long total = (long long)B * 2 * h * (2 * w / 4);
  const int g = grid_for(total, 256);
  if (dtype == B200SEG_BF16 && C <= 12)
    launch_pdl(upsample2x_ac_kernel<bf16, float, 4, 12, true>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const bf16*)logits, nullptr, mask, B, h, w, C);
  else if (dtype == B200SEG_BF16)
    launch_pdl(upsample2x_ac_kernel<bf16, float, 4, 16, true>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const bf16*)logits, nullptr, mask, B, h, w, C);
  else if (dtype == B200SEG_F32)
    launch_pdl(upsample2x_ac_kernel<float, float, 4, 16, true>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const float*)logits, nullptr, mask, B, h, w, C);
  else return set_error(-1, "upsample2x_ac_argmax: bad dtype");
  return check_launch("upsample2x_ac_argmax");
}

int b200seg_nhwc_to_nchw(const void* x, int dtype, int ldc, void* out, int out_dtype, int B, int H, int W, int C,
                         b200seg_stream_t s) {
  B200_REQUIRE(C >= 1 && ldc >= C && B > 0 && H > 0 && W > 0, "nhwc_to_nchw: bad shape");
  cudaStream_t st = (cudaStream_t)s;
  const int g = grid_for((long long)B * H * W, 256);
#define LAUNCH(T, TO) launch_pdl(nhwc_to_nchw_kernel<T, TO>, dim3((unsigned)g), dim3((unsigned)256), (size_t)0, st, (const T*)x, ldc, (TO*)out, B, H, W, C)
  if (dtype == B200SEG_BF16 && out_dtype == B200SEG_BF16) LAUNCH(bf16, bf16);
  else if (dtype == B200SEG_BF16 && out_dtype == B200SEG_F32) LAUNCH(bf16, float);
  else if (dtype == B200SEG_F32 && out_dtype == B200SEG_F32) LAUNCH(float, float);
  else if (dtype == B200SEG_F32 && out_dtype == B200SEG_BF16) LAUNCH(float, bf16);
  else return set_error(-1, "nhwc_to_nchw: bad dtypes");
#undef LAUNCH
  return check_launch("nhwc_to_nchw");
}

int b200seg_maxpool2x2(const void* x, void* y, int dtype, int B, int H, int W, int C, b200seg_stream_t s) {
  const int vn = dtype == B200SEG_BF16 ? 8 : 4;
  B200_REQUIRE(dtype == B200SEG_BF16 || dtype == B200SEG_F32, "maxpool2x2: bad dtype");
  B200_REQUIRE(C % vn == 0 && H % 2 == 0 && W % 2 == 0 && B > 0 && H > 0 && W > 0, "maxpool2x2: bad shape C=%d H=%d W=%d", C, H, W);
  cudaStream_t st = (cudaStream_t)s;
  const long long total = (long long)B * (H / 2) * (W / 2) * (C / vn);
  if (dtype == B200SEG_BF16)
    launch_pdl(maxpool2x2_kernel<bf16>, dim3((unsigned)grid_for(total, 256)), dim3((unsigned)256), (size_t)0, st, (const bf16*)x, (bf16*)y, B, H, W, C);
  else
    launch_pdl(maxpool2x2_kernel<float>, dim3((unsigned)grid_for(total, 256)), dim3((unsigned)256), (size_t)0, st, (const float*)x, (float*)y, B, H, W, C);
  return check_launch("maxpool2x2");
}

}  // extern "C"
