// conv_rs.cu -- 3x3 convolution with FEW output channels as a "row-stacked" implicit GEMM on tcgen05.
//
// Why: the cost of one tcgen05.mma (M = 128, K = 16) is max(N/2, 32 + N/4) cycles (tools/mma_probe.py): below N = 128 it
// barely depends on N, so conv_tc's schedule for Cout = 32 -- 9 taps x K/16 instructions of N = 32 per 128 pixels, 40 cycles
// each -- is bound by the instruction COUNT (up4.conv.0: 45 MMAs per tile, issue floor 101 us, measured 202 us) and reads
// every input row from shared memory nine times.  Here the three vertical taps are stacked along N instead:
//
//     D_r[p, kh*CN + co] = sum_{kw, ci} X[r, p + kw - 1, ci] * W[co][kh][kw][ci]          (one accumulator per INPUT row r)
//     out[h, p, co]      = D_{h-1}[p, 0*CN + co] + D_h[p, 1*CN + co] + D_{h+1}[p, 2*CN + co]
//
// One input row costs 3 x K/16 instructions of N = 3*CN (56 cycles for CN = 32) instead of 9 x K/16 of N = CN per output row:
// 2.1x fewer tensor-pipe cycles, 3x fewer shared-memory operand reads, and each input row is fetched once per strip.  The sum
// over the three accumulators has the same pixel (TMEM lane) in all terms, so the epilogue thread of a pixel column keeps two
// running rows in registers and finishes one output row per input row -- no cross-lane traffic.
//
// Persistent CTAs split the flattened (image, column tile, row) space evenly (a CTA's range may span strips; every
// contiguous run of rows pays two halo rows).  Warp roles as in conv_tc: warp 0 TMA producer (one 130-pixel halo box per
// input row and 64-channel chunk, borders = TMA zero fill), warp 1 TMEM owner + MMA issuer (weights resident in shared
// memory, 3 x 3 x chunks tiles of [3*CN][64]), warps 2..5 epilogue.  Two TMEM accumulators: the MMAs of row r+1 overlap the
// epilogue of row r.
//
// Two-source input (b200seg_conv_rs_cat): cat([S, U], channel) read from the two dense tensors as in conv_tc -- chunks
// 0 .. ks-1 from S, the rest from U, weight columns at Cs + 64(c - ks) for a U chunk (see conv_tc.cu).
#include "common.cuh"

namespace b200 {

struct ConvRsArgs {
  const float* bias;
  const void* res;     // added after the activation (dgrad accumulation / shortcut), or NULL
  void* y;
  int Cin, Cout;
  int W, H, B;
  int BW, tiles_w;
  int k_chunks, stages;   // k_chunks = ceil(Cs / 64) + ceil((Cin - Cs) / 64)
  int Cs, ks;             // two-source input: channels of S and its chunk count; 0 = one source
  int act;
  long long total_rows;   // B * tiles_w * H
};

constexpr int RS_THREADS = 192;
constexpr int RS_HALO_BYTES = 17 * 1024;   // 130 rows x 128 B rounded up to the 1024-B swizzle atom

// Walks the input rows of the range [g0, g1) of flattened output rows: calls f(strip, r, valid, emit, new_run) for every
// input row r in [ha-1, hb] of every contiguous run [ha, hb) of one strip; emit = output row r-1 belongs to the run.
template <typename F>
__device__ __forceinline__ void rs_walk(long long g0, long long g1, int H, F&& f) {
  long long g = g0;
  while (g < g1) {
    const long long strip = g / H;
    const int ha = (int)(g - strip * H);
    const int hb = (int)min((long long)H, (long long)ha + (g1 - g));
    for (int r = ha - 1; r <= hb; ++r) f(strip, r, r >= 0 && r < H, r - 1 >= ha, r == ha - 1);
    g += hb - ha;
  }
}

// CAT: two-source input (Cs > 0); the one-source instantiation carries no per-chunk source selection
template <int CN, bool CAT>
__global__ void __launch_bounds__(RS_THREADS, CN <= 32 ? 2 : 1)
conv_rs_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmS, const ConvRsArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = CAT ? a.ks : 0, Cs = CAT ? a.Cs : 0;
  constexpr int NACC = 3 * CN;                    // accumulator columns per input row
  constexpr int B_TILE = NACC * 128;              // one (chunk, kw) weight tile: [3*CN rows][64 k] bf16

  uint8_t* sA = smem;
  uint8_t* sB = sA + a.stages * RS_HALO_BYTES;
  float* sBias = reinterpret_cast<float*>(sB + a.k_chunks * 3 * B_TILE);
  uint64_t* full = reinterpret_cast<uint64_t*>(sBias + CN);
  uint64_t* empty = full + 8;
  uint64_t* acc_full = empty + 8;      // [2]
  uint64_t* acc_empty = acc_full + 2;  // [2]
  uint64_t* b_full = acc_empty + 2;    // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_full + 1);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (CAT) tma_prefetch_desc(&tmS);
    for (int i = 0; i < a.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 128); }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < CN; i += RS_THREADS) sBias[i] = (a.bias && i < a.Cout) ? a.bias[i] : 0.f;
  constexpr uint32_t TMEM_COLS = 2 * NACC <= 32 ? 32 : 2 * NACC <= 64 ? 64 : 2 * NACC <= 128 ? 128 : 2 * NACC <= 256 ? 256 : 512;
  if (warp == 1) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const long long g0 = a.total_rows * blockIdx.x / gridDim.x, g1 = a.total_rows * (blockIdx.x + 1) / gridDim.x;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      mbar_arrive_expect_tx(b_full, (uint32_t)(a.k_chunks * 3 * B_TILE));
      for (int c = 0; c < a.k_chunks; ++c)
        for (int kw = 0; kw < 3; ++kw)
          for (int kh = 0; kh < 3; ++kh)          // rows [kh*CN, +CN) of tile (c, kw) <- W[:, tap kh*3+kw, chunk c]
            tma_load_3d(sB + (c * 3 + kw) * B_TILE + kh * CN * 128, &tmB, b_full, CAT && c < ks ? c * 64 : Cs + (c - ks) * 64,
                        kh * 3 + kw, 0);
    }
    int s = 0;
    uint32_t ph = 0;
    rs_walk(g0, g1, a.H, [&](long long strip, int r, bool valid, bool, bool) {
      if (!valid) return;
      const int w0 = (int)(strip % a.tiles_w) * a.BW, bb = (int)(strip / a.tiles_w);
      for (int c = 0; c < a.k_chunks; ++c) {
        mbar_wait(&empty[s], ph ^ 1u, 1);
        if (lane == 0) {
          mbar_arrive_expect_tx(&full[s], 130u * 128u);
          const bool sk = CAT && c < ks;
          tma_load_4d(sA + s * RS_HALO_BYTES, sk ? &tmS : &tmA, &full[s], sk ? c * 64 : (c - ks) * 64, w0 - 1, r, bb);
        }
        __syncwarp();
        if (++s == a.stages) { s = 0; ph ^= 1u; }
      }
    });
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t idesc = umma_idesc_bf16(128, NACC);
    const uint32_t desc_hi = (uint32_t)(umma_desc_k128(0) >> 32);
    const uint32_t a_lo0 = (uint32_t)umma_desc_k128(smem_u32(sA));
    const uint32_t b_lo0 = (uint32_t)umma_desc_k128(smem_u32(sB));
    mbar_wait(b_full, 0, 5);
    int s = 0, nrow = 0;
    uint32_t ph = 0;
    rs_walk(g0, g1, a.H, [&](long long, int, bool valid, bool, bool) {
      if (!valid) return;
      const int ab = nrow & 1;
      const uint32_t aph = (uint32_t)(nrow >> 1) & 1u;
      ++nrow;
      mbar_wait(&acc_empty[ab], aph ^ 1u, 6);
      tc_fence_after();
      const uint32_t tacc = tmem_base + (uint32_t)(ab * NACC);
      uint32_t first = 0;
      for (int c = 0; c < a.k_chunks; ++c) {
        const int krem = CAT && c < ks ? Cs - c * 64 : a.Cin - Cs - (c - ks) * 64;   // channels left in the chunk's source
        const int ksteps = (min(64, krem) + 15) >> 4;
        const uint32_t a_lo = a_lo0 + (uint32_t)s * (RS_HALO_BYTES >> 4);
        mbar_wait(&full[s], ph, 2);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            const uint32_t al = a_lo + (uint32_t)kw * 8u;                       // +128 B: one pixel to the right
            const uint32_t bl = b_lo0 + (uint32_t)(c * 3 + kw) * (B_TILE >> 4);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k < ksteps) { umma_bf16_lohi(tacc, al + 2u * k, bl + 2u * k, desc_hi, idesc, first); first = 1u; }
          }
          umma_commit(&empty[s]);
          if (c == a.k_chunks - 1) umma_commit(&acc_full[ab]);
        }
        __syncwarp();
        if (++s == a.stages) { s = 0; ph ^= 1u; }
      }
    });
  } else {
    // ================= epilogue (warps 2..5): thread = pixel column =================
    const int q = warp & 3;
    const int p = q * 32 + lane;
    const float act_lo = (a.act != B200SEG_ACT_NONE) ? 0.f : -INFINITY;
    const float act_hi = (a.act == B200SEG_ACT_RELU6) ? 6.f : INFINITY;
    const bool vec32 = (a.Cout & 15) == 0;
    float run0[CN], run1[CN];       // partial sums of output rows r and r+1 (see header)
    int nrow = 0;
    rs_walk(g0, g1, a.H, [&](long long strip, int r, bool valid, bool emit, bool new_run) {
      const int w0 = (int)(strip % a.tiles_w) * a.BW, bb = (int)(strip / a.tiles_w);
      if (new_run) {
#pragma unroll
        for (int i = 0; i < CN; ++i) { run0[i] = 0.f; run1[i] = 0.f; }
      }
      const bool px_ok = p < a.BW && w0 + p < a.W;
      const long long pix = ((long long)bb * a.H + (r - 1)) * a.W + (w0 + p);
      const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(a.res) + pix * a.Cout;
      __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(a.y) + pix * a.Cout;
      int ab = 0;
      if (valid) {
        ab = nrow & 1;
        const uint32_t aph = (uint32_t)(nrow >> 1) & 1u;
        ++nrow;
        mbar_wait(&acc_full[ab], aph, 3);
        tc_fence_after();
      }
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * NACC);
#pragma unroll
      for (int j = 0; j < CN / 16; ++j) {
        uint32_t d0[16], d1[16], d2[16];
        if (valid) {
          tmem_ld16(trow + (uint32_t)(16 * j), d0);                // kh = 0 -> output row r+1
          tmem_ld16(trow + (uint32_t)(CN + 16 * j), d1);           // kh = 1 -> output row r
          tmem_ld16(trow + (uint32_t)(2 * CN + 16 * j), d2);       // kh = 2 -> output row r-1
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) { d0[i] = 0u; d1[i] = 0u; d2[i] = 0u; }
        }
        float f[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          f[i] = run0[16 * j + i] + __uint_as_float(d2[i]);
          run0[16 * j + i] = run1[16 * j + i] + __uint_as_float(d1[i]);
          run1[16 * j + i] = __uint_as_float(d0[i]);
        }
        if (emit && px_ok && 16 * j < a.Cout) {
          const bool c_ok1 = 16 * j + 8 < a.Cout;                  // Cout % 8 == 0
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = fminf(fmaxf(f[i] + sBias[16 * j + i], act_lo), act_hi);
          if (a.res != nullptr) {
            const uint4 u0 = __ldg(reinterpret_cast<const uint4*>(rp + 16 * j));
            uint4 u1 = make_uint4(0, 0, 0, 0);
            if (c_ok1) u1 = __ldg(reinterpret_cast<const uint4*>(rp + 16 * j + 8));
            const uint32_t t[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) { f[2 * i] += bf16lo(t[i]); f[2 * i + 1] += bf16hi(t[i]); }
          }
          uint32_t o[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] = pack_bf16x2(f[2 * i], f[2 * i + 1]);
          if (vec32) {
            asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(yp + 16 * j), "r"(o[0]), "r"(o[1]),
                         "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7])
                         : "memory");
          } else {
            *reinterpret_cast<uint4*>(yp + 16 * j) = make_uint4(o[0], o[1], o[2], o[3]);
            if (c_ok1) *reinterpret_cast<uint4*>(yp + 16 * j + 8) = make_uint4(o[4], o[5], o[6], o[7]);
          }
        }
      }
      if (valid) {
        tc_fence_before();
        mbar_arrive(&acc_empty[ab]);
      }
    });
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int CN, bool CAT>
static int launch_conv_rs(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmS, ConvRsArgs a, int flags,
                          cudaStream_t stream) {
  const int b_all = a.k_chunks * 3 * (3 * CN * 128);
  const int fixed = b_all + CN * 4 + 256 + 1024 /*align slack*/;
  const int tmem_cols = 2 * 3 * CN <= 256 ? 256 : 512;
  int per_sm = (tmem_cols <= 256 && CN <= 32) ? 2 : 1;
  // two CTAs per SM (two issuers, two epilogues) whenever a 2-stage ring still fits: measured faster than one CTA with a
  // deep ring on every up4 shape (tools/kbench_rs.py: 80->32 114 vs 124 us, 32->32 58 vs 82 us at B=64)
  int stages = (227 * 1024 / per_sm - 1024 - fixed) / RS_HALO_BYTES;
  if (per_sm == 2 && stages < 2) { per_sm = 1; stages = (227 * 1024 - 1024 - fixed) / RS_HALO_BYTES; }
  if ((flags >> 20) & 3) { per_sm = (flags >> 20) & 3; stages = (227 * 1024 / per_sm - 1024 - fixed) / RS_HALO_BYTES; }
  if (stages > 8) stages = 8;
  if ((flags >> 16) & 0xf) stages = min(stages, (flags >> 16) & 0xf);
  B200_REQUIRE(stages >= 2, "conv_rs: weights do not leave room for a load ring (Cin=%d Cout=%d)", a.Cin, a.Cout);
  a.stages = stages;
  const int smem = fixed + stages * RS_HALO_BYTES;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_rs_kernel<CN, CAT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return set_error((int)e, "conv_rs: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr = true;
  }
  long long grid = (long long)sm_count() * per_sm;
  if ((flags >> 8) & 0xff) grid = (long long)((flags >> 8) & 0xff) * 4;
  if (grid > a.total_rows) grid = a.total_rows;
  conv_rs_kernel<CN, CAT><<<(unsigned)grid, RS_THREADS, (size_t)smem, stream>>>(tmA, tmB, tmS, a);
  return check_launch("conv_rs");
}

}  // namespace b200

using namespace b200;

static int rs_supported(int H, int W, int Cs, int Cin, int Cout) {
  const int cn = (Cout + 15) & ~15;
  const int k_chunks = (Cs + 63) / 64 + (Cin - Cs + 63) / 64;
  // cn = 80: the data gradient of up4.conv.0 (32 -> 80 channels): N = 240, two accumulators = 480 TMEM columns, the
  // epilogue's two running rows take 160 registers (one CTA per SM, 255 registers per thread)
  return (cn == 16 || cn == 32 || cn == 80) && W >= 96 && H >= 3 && Cin % 8 == 0 && Cout % 8 == 0 &&
         k_chunks * 3 * (3 * cn * 128) <= 120 * 1024;
}

// 1 if b200seg_conv_rs supports the shape (the engine asks before choosing it over b200seg_conv_tc)
extern "C" int b200seg_conv_rs_supported(int H, int W, int Cin, int Cout) { return rs_supported(H, W, 0, Cin, Cout); }

// the same for b200seg_conv_rs_cat (skip S with Cs channels + U with Cu channels)
extern "C" int b200seg_conv_rs_cat_supported(int H, int W, int Cs, int Cu, int Cout) {
  return Cs >= 0 && Cs % 8 == 0 && Cu > 0 && rs_supported(H, W, Cs, Cs + Cu, Cout);
}

// 3x3, pad 1, stride 1, bf16 NHWC, few output channels (see b200seg_conv_rs_supported).  Same operands and results as
// b200seg_conv_tc(taps = 9): w bf16 [Cout][9][Cin], b f32 [Cout] or NULL, res added after the activation.
// flags: bits 8..15 grid/4, bits 16..19 max ring stages, bits 20..21 CTAs per SM (0 = auto).
static int conv_rs_run(const void* skip, int Cs, const void* x, const void* w, const float* bias, const void* res, void* y,
                       int B, int H, int W, int Cin, int Cout, int act, int flags, cudaStream_t stream) {
  const int Cu = Cin - Cs;
  ConvRsArgs a;
  a.bias = bias; a.res = res; a.y = y;
  a.Cin = Cin; a.Cout = Cout; a.W = W; a.H = H; a.B = B;
  a.BW = W < 128 ? W : 128;
  a.tiles_w = (W + a.BW - 1) / a.BW;
  a.k_chunks = (Cs + 63) / 64 + (Cu + 63) / 64;
  a.Cs = Cs; a.ks = (Cs + 63) / 64;
  a.act = act;
  a.total_rows = (long long)B * a.tiles_w * H;
  const int cn = (Cout + 15) & ~15;
  CUtensorMap tmA, tmB, tmS;
  for (int src = 0; src < (Cs ? 2 : 1); ++src) {
    const uint64_t c = (uint64_t)(src ? Cs : Cu);
    uint64_t dims[4] = {c, (uint64_t)W, (uint64_t)H, (uint64_t)B};
    uint64_t str[3] = {c * 2, c * 2 * W, c * 2 * W * H};
    uint32_t box[4] = {64, 130, 1, 1};
    int rc = make_tmap_bf16(src ? &tmS : &tmA, src ? skip : x, 4, dims, str, box, 1, nullptr);
    if (rc) return rc;
  }
  if (!Cs) tmS = tmA;
  {
    uint64_t dims[3] = {(uint64_t)Cin, 9, (uint64_t)Cout};
    uint64_t str[2] = {(uint64_t)Cin * 2, (uint64_t)Cin * 2 * 9};
    uint32_t box[3] = {64, 1, (uint32_t)cn};
    int rc = make_tmap_bf16(&tmB, w, 3, dims, str, box, 1, nullptr);
    if (rc) return rc;
  }
  if (Cs) {
    if (cn == 16) return launch_conv_rs<16, true>(tmA, tmB, tmS, a, flags, stream);
    if (cn == 80) return launch_conv_rs<80, true>(tmA, tmB, tmS, a, flags, stream);
    return launch_conv_rs<32, true>(tmA, tmB, tmS, a, flags, stream);
  }
  if (cn == 16) return launch_conv_rs<16, false>(tmA, tmB, tmS, a, flags, stream);
  if (cn == 80) return launch_conv_rs<80, false>(tmA, tmB, tmS, a, flags, stream);
  return launch_conv_rs<32, false>(tmA, tmB, tmS, a, flags, stream);
}

extern "C" int b200seg_conv_rs(const void* x, const void* w, const float* bias, const void* res, void* y, int B, int H,
                               int W, int Cin, int Cout, int act, int flags, b200seg_stream_t s) {
  B200_REQUIRE(x && w && y && B > 0, "conv_rs: bad arguments");
  B200_REQUIRE(b200seg_conv_rs_supported(H, W, Cin, Cout), "conv_rs: unsupported shape H=%d W=%d Cin=%d Cout=%d", H, W, Cin, Cout);
  return conv_rs_run(nullptr, 0, x, w, bias, res, y, B, H, W, Cin, Cout, act, flags, (cudaStream_t)s);
}

// two-source input: cat([skip [B,H,W,Cs], x [B,H,W,Cu]], channel), w bf16 [Cout][9][Cs + Cu]
extern "C" int b200seg_conv_rs_cat(const void* skip, const void* x, const void* w, const float* bias, const void* res,
                                   void* y, int B, int H, int W, int Cs, int Cu, int Cout, int act, int flags,
                                   b200seg_stream_t s) {
  B200_REQUIRE(x && w && y && B > 0 && (skip || !Cs), "conv_rs_cat: bad arguments");
  B200_REQUIRE(b200seg_conv_rs_cat_supported(H, W, Cs, Cu, Cout), "conv_rs_cat: unsupported shape H=%d W=%d Cs=%d Cu=%d Cout=%d",
               H, W, Cs, Cu, Cout);
  return conv_rs_run(skip, Cs, x, w, bias, res, y, B, H, W, Cs + Cu, Cout, act, flags, (cudaStream_t)s);
}
