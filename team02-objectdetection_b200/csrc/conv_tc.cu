// conv_tc.cu -- dense 1x1 / 3x3 convolution as an implicit GEMM on the 5th-gen tensor cores.
//
//   D[128 pixels, N couts] (fp32, TMEM) = sum over (tap, cin-chunk) A[128, 64] * B[N, 64]^T
//
// Persistent, warp-specialised kernel: one CTA per SM slot loops over output tiles; three
// pipelines run concurrently
//     TMA producer --(smem ring: full/empty)--> MMA issuer --(TMEM x2: acc_full/acc_empty)--> epilogue
// so the loads of tile i+1, the MMAs of tile i and the epilogue/stores of tile i-1 overlap.
//
// A operand (activations, NHWC bf16) -- two addressing modes, both pure TMA:
//   TAP   : a 4-D tiled tensor map (C, W, H, B), box {64, BW, BH, 1}; each 3x3 tap is the same box
//           shifted by (dw, dh).  Zero padding, ragged borders and the Cin tail are TMA OOB zero fill.
//           1x1 convs use it with the pixels flattened to one axis (box {64,128,1,1}).
//   HALO  : (3x3, tiles = 128 consecutive pixels of one image row) one box {64, 130, 1, 1} per input
//           row h-1, h, h+1 is loaded ONCE per cin-chunk; the three horizontal taps are the same
//           shared-memory tile read through UMMA descriptors whose start address is advanced by
//           dw*128 bytes (descriptor base_offset = dw keeps the 128-byte swizzle phase right).
//           L2->smem traffic for A drops from 9x to 3 x 130/128.
// B operand (weights bf16 [Cout][taps][Cin]): 3-D map, box {64,1,N}; when all taps/chunks of the N
// tile fit in shared memory they are loaded once per CTA ("resident") instead of once per tile.
//
// Two-source A (the decoder's first 3x3 conv of an up stage): the input is cat([S, U], channel) with S
// [B][H][W][Cs] and U [B][H][W][Cu] kept as two dense tensors.  K chunks 0 .. ks-1 (ks = ceil(Cs/64)) load
// from a map over S at channel 64c, the rest from the map over U at channel 64(c-ks); the weight box of a U
// chunk starts at channel Cs + 64(c-ks).  In a narrow skip chunk the weight columns past Cs belong to U, but
// they meet S's out-of-bounds zero fill and add exact zeros; the chunk issues ceil((Cs-64c)/16) k-steps, so
// the issued MMAs are those of the concatenated tensor.  Cs = 0 is the single-tensor path.
//
// Epilogue: TMEM -> registers (tcgen05.ld 32x32b.x16, double-buffered) -> +bias -> ReLU/ReLU6 -> +residual
// -> bf16 -> one 256-bit global store per 16 channels (thread = pixel, so each store is a full 32-byte
// sector of that pixel's NHWC row).  An alternative epilogue (flag bit0) goes through a 128B-swizzled
// staging tile and a TMA store; it is slower because the store queues behind the prefetched loads in the
// same TMA unit and the staging buffer cannot be reused until the store has drained.
//
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer,
// warps 2..5 = epilogue (TMEM lane quadrant = warp_id % 4).
#include "common.cuh"

namespace b200 {

struct ConvTcArgs {
  const float* bias;
  const void* res;   // residual, read straight from global in the epilogue (or NULL)
  void* y;
  int taps, Cin, Cout;
  int W, H, B;       // geometry the tile scheduler walks (1x1: W = #pixels, H = B = 1)
  int BW, BH;        // M tile = BH rows x BW columns of pixels, BW*BH <= 128
  int tiles_w, tiles_h;
  int block_n, n_tiles;
  int k_chunks;      // ceil(Cs / 64) + ceil((Cin - Cs) / 64)
  int Cs, ks;        // two-source A: channels of S and its chunk count ceil(Cs / 64); 0 = one source
  int stages;
  int act;
  int tma_store;     // epilogue: 0 = 256-bit stores straight from registers, 1 = smem staging + TMA store
  int tmem_cols;
  int halo;          // A addressing mode (see above)
  int b_resident;    // weights loaded once per CTA
  int pdl_early;     // trigger dependents at kernel start (else just before the final barrier)
  int n_sbuf;        // staging buffers (1 or 2)
  int halo_bo;       // HALO: put the swizzle phase of the shifted start address into descriptor.base_offset
  int dw;            // depthwise mode: B is block-diagonal, the only K chunk of N tile j is channel chunk j
  int stride;        // 1, or 2 (TAP mode only; the A tensor map then carries elementStrides = 2)
  int a_stage_bytes, b_stage_bytes;
  int mpair;         // M tiles (128 pixels each) per work item that share every B stage (1 or 2)
  int acc_bufs;      // TMEM accumulator sets: 2 = epilogue overlaps the next item's MMAs, 1 = no room
  long long m_tiles; // real pixel tiles; work items = ceil(m_tiles / mpair) * n_tiles
  long long total_tiles;
};

constexpr int TC_THREADS = 192;
constexpr int TILE_BYTES = 128 * 128;   // 128 rows x 64 bf16
constexpr int HALO_BYTES = 17 * 1024;   // 130 rows x 128 B rounded up to the 1024-B swizzle atom

__device__ __forceinline__ uint64_t umma_desc_k128_off(uint32_t smem_addr) {
  // start address not 1024-aligned: base_offset = (addr >> 7) & 7 (PTX ISA, tcgen05 matrix descriptor)
  return umma_desc_k128(smem_addr) | ((uint64_t)((smem_addr >> 7) & 7u) << 49);
}

// CAT: two-source A (Cs > 0).  The one-source instantiation carries none of the per-chunk source selection.
template <int MPAIR, bool CAT>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmS, const ConvTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = CAT ? a.ks : 0, Cs = CAT ? a.Cs : 0;
  const int n_boxes = (a.block_n + 63) >> 6;
  const int kb_per_tile = a.halo ? a.k_chunks * 3 : a.k_chunks * a.taps;
  const int b_tiles_resident = a.taps * a.k_chunks;
  const int b_tile_bytes = a.block_n * 128;

  uint8_t* sA = smem;
  const int a_stride = MPAIR * a.a_stage_bytes;      // one ring slot holds the A tiles of all paired M tiles
  uint8_t* sB = sA + a.stages * a_stride;
  uint8_t* sOut = sB + (a.b_resident ? b_tiles_resident * b_tile_bytes : a.stages * a.b_stage_bytes);
  float* sBias = reinterpret_cast<float*>(sOut + a.n_sbuf * n_boxes * TILE_BYTES);
  uint64_t* full = reinterpret_cast<uint64_t*>(sBias + 256);
  uint64_t* empty = full + 8;
  uint64_t* acc_full = empty + 8;      // [2]
  uint64_t* acc_empty = acc_full + 2;  // [2]
  uint64_t* b_full = acc_empty + 2;    // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(b_full + 1);

  if (a.pdl_early) pdl_trigger();      // the next kernel's prologue may overlap this kernel's tail
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (CAT) tma_prefetch_desc(&tmS);
    if (a.tma_store) tma_prefetch_desc(&tmC);
    for (int i = 0; i < a.stages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 128);
    }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)a.tmem_cols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int rows = a.BW * a.BH;

  if (warp == 0) {
    // ================= TMA producer =================
    if (a.b_resident && lane == 0) {
      mbar_arrive_expect_tx(b_full, (uint32_t)(b_tiles_resident * b_tile_bytes));
      for (int t = 0; t < a.taps; ++t)
        for (int c = 0; c < a.k_chunks; ++c)
          tma_load_3d(sB + (t * a.k_chunks + c) * b_tile_bytes, &tmB, b_full, CAT && c < ks ? c * 64 : Cs + (c - ks) * 64, t, 0);
    }
    pdl_wait();         // weights are static; activations come from the previous kernel
    int s = 0;
    uint32_t ph = 0;
    const int n_outer = a.halo ? a.k_chunks : a.taps;      // HALO: chunks x 3 rows;  TAP: taps x chunks
    const int n_inner = a.halo ? 3 : a.k_chunks;
    const uint32_t tx_bytes = a.halo ? (uint32_t)MPAIR * 130u * 128u + (a.b_resident ? 0u : 3u * (uint32_t)b_tile_bytes)
                                     : (uint32_t)(MPAIR * rows * 128 + (a.b_resident ? 0 : b_tile_bytes));
    for (long long tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
      const int n_tile = (int)(tile % a.n_tiles);
      const int n0 = n_tile * a.block_n;
      int w0v[MPAIR], h0v[MPAIR], bbv[MPAIR];
#pragma unroll
      for (int j = 0; j < MPAIR; ++j) {       // a pair index past the last real tile decodes to bb >= B: all OOB
        long long mt = (tile / a.n_tiles) * MPAIR + j;
        w0v[j] = (int)(mt % a.tiles_w) * a.BW; mt /= a.tiles_w;
        h0v[j] = (int)(mt % a.tiles_h) * a.BH;
        bbv[j] = (int)(mt / a.tiles_h);
      }
      for (int o = 0; o < n_outer; ++o) {
        for (int i = 0; i < n_inner; ++i) {
          mbar_wait(&empty[s], ph ^ 1u, 1);
          if (lane == 0) {
            mbar_arrive_expect_tx(&full[s], tx_bytes);
            if (a.halo) {
              const int chunk = o, dh = i;
              const int ach = a.dw ? n_tile : chunk;           // channel chunk of the activations
              const bool sk = CAT && ach < ks;                 // chunk of the skip source
              const CUtensorMap* tmX = sk ? &tmS : &tmA;
              const int xc = sk ? ach * 64 : (ach - ks) * 64, wc = sk ? chunk * 64 : Cs + (chunk - ks) * 64;
#pragma unroll
              for (int j = 0; j < MPAIR; ++j)
                tma_load_4d(sA + s * a_stride + j * a.a_stage_bytes, tmX, &full[s], xc, w0v[j] - 1,
                            h0v[j] + dh - 1, bbv[j]);
              if (!a.b_resident)
                for (int dw = 0; dw < 3; ++dw)
                  tma_load_3d(sB + s * a.b_stage_bytes + dw * b_tile_bytes, &tmB, &full[s], a.dw ? 0 : wc,
                              dh * 3 + dw, n0);
            } else {
              const int tap = o, chunk = i;
              const int ach = a.dw ? n_tile : chunk;
              const bool sk = CAT && ach < ks;
              const CUtensorMap* tmX = sk ? &tmS : &tmA;
              const int xc = sk ? ach * 64 : (ach - ks) * 64, wc = sk ? chunk * 64 : Cs + (chunk - ks) * 64;
              int dw = 0, dh = 0;
              if (a.taps == 9) { dh = tap / 3 - 1; dw = tap - (dh + 1) * 3 - 1; }
#pragma unroll
              for (int j = 0; j < MPAIR; ++j)
                tma_load_4d(sA + s * a_stride + j * a.a_stage_bytes, tmX, &full[s], xc, w0v[j] * a.stride + dw,
                            h0v[j] * a.stride + dh, bbv[j]);
              if (!a.b_resident)
                tma_load_3d(sB + s * a.b_stage_bytes, &tmB, &full[s], a.dw ? 0 : wc, tap, n0);
            }
          }
          __syncwarp();
          if (++s == a.stages) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    // One thread issues every tcgen05.mma of the CTA, so its scalar instruction count per MMA bounds the
    // tile rate of the short-K layers: descriptors are kept as {lo,hi} 32-bit halves (hi is constant), the
    // k loop is fully unrolled, and ring indices are carried incrementally (no div/mod).
    const uint32_t idesc = umma_idesc_bf16(128, a.block_n);
    const uint32_t desc_hi = (uint32_t)(umma_desc_k128(0) >> 32);
    const uint32_t a_lo0 = (uint32_t)umma_desc_k128(smem_u32(sA));      // low word for stage 0
    const uint32_t b_lo0 = (uint32_t)umma_desc_k128(smem_u32(sB));
    const uint32_t a_stage16 = (uint32_t)a_stride >> 4, a_tile16 = (uint32_t)a.a_stage_bytes >> 4;
    const uint32_t b_stage16 = (uint32_t)a.b_stage_bytes >> 4;
    const uint32_t b_tile16 = (uint32_t)b_tile_bytes >> 4;
    const int n_outer = a.halo ? a.k_chunks : a.taps;
    const int n_inner = a.halo ? 3 : a.k_chunks;
    if (a.b_resident) mbar_wait(b_full, 0, 5);
    int s = 0;
    uint32_t ph = 0;
    int it = 0;
    for (long long tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++it) {
      const int ab = a.acc_bufs == 2 ? (it & 1) : 0;
      const uint32_t aph = (uint32_t)(a.acc_bufs == 2 ? (it >> 1) : it) & 1u;
      mbar_wait(&acc_empty[ab], aph ^ 1u, 6);     // epilogue has drained this accumulator set
      tc_fence_after();
      const uint32_t tacc0 = tmem_base + (uint32_t)(ab * MPAIR * a.block_n);
      const int n_tile = a.dw ? (int)(tile % a.n_tiles) : 0;
      uint32_t first = 0;                           // 0 for the very first k-block of the item (overwrite), then 1
      for (int o = 0; o < n_outer; ++o) {
        for (int i = 0; i < n_inner; ++i) {
          const int chunk = a.halo ? o : i;
          const int cc = a.dw ? n_tile : chunk;       // channels left in this chunk's source (skip S, or U / the single input)
          const int krem = CAT && cc < ks ? Cs - cc * 64 : a.Cin - Cs - (cc - ks) * 64;
          const int ksteps = (min(64, krem) + 15) >> 4;
          const uint32_t a_lo = a_lo0 + (uint32_t)s * a_stage16;
          mbar_wait(&full[s], ph, 2);
          tc_fence_after();
          if (elect_one()) {
            if (a.halo) {
              const int dh = i;
#pragma unroll
              for (int j = 0; j < MPAIR; ++j) {
                const uint32_t tacc = tacc0 + (uint32_t)(j * a.block_n);
                uint32_t fj = first;
#pragma unroll
                for (int dw = 0; dw < 3; ++dw) {
                  const int tap = dh * 3 + dw;
                  const uint32_t al = a_lo + (uint32_t)j * a_tile16 + (uint32_t)dw * 8u;   // +128 B: one pixel to the right
                  const uint32_t bl = a.b_resident ? b_lo0 + (uint32_t)(tap * a.k_chunks + chunk) * b_tile16
                                                   : b_lo0 + (uint32_t)s * b_stage16 + (uint32_t)dw * b_tile16;
#pragma unroll
                  for (int k = 0; k < 4; ++k)
                    if (k < ksteps) { umma_bf16_lohi(tacc, al + 2u * k, bl + 2u * k, desc_hi, idesc, fj); fj = 1u; }
                }
              }
            } else {
              const int tap = o;
              const uint32_t bl = a.b_resident ? b_lo0 + (uint32_t)(tap * a.k_chunks + chunk) * b_tile16
                                               : b_lo0 + (uint32_t)s * b_stage16;
#pragma unroll
              for (int j = 0; j < MPAIR; ++j) {
                const uint32_t tacc = tacc0 + (uint32_t)(j * a.block_n);
                const uint32_t al = a_lo + (uint32_t)j * a_tile16;
                uint32_t fj = first;
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (k < ksteps) { umma_bf16_lohi(tacc, al + 2u * k, bl + 2u * k, desc_hi, idesc, fj); fj = 1u; }
              }
            }
            first = 1u;
            umma_commit(&empty[s]);
            if (o == n_outer - 1 && i == n_inner - 1) umma_commit(&acc_full[ab]);
          }
          __syncwarp();
          if (++s == a.stages) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else {
    // ================= epilogue (warps 2..5) =================
    const int et = threadIdx.x - 64;
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int hl = r / a.BW, wl = r - hl * a.BW;
    const float act_lo = (a.act != B200SEG_ACT_NONE) ? 0.f : -INFINITY;
    const float act_hi = (a.act == B200SEG_ACT_RELU6) ? 6.f : INFINITY;
    const bool vec32 = (a.Cout & 15) == 0;     // pixel pitch is a multiple of 32 B -> 256-bit accesses
    pdl_wait();         // residual reads / output writes must follow the previous kernel
    int it = 0;
    int cur_n_tile = -1;
    for (long long tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x, ++it) {
      const int n_tile = (int)(tile % a.n_tiles);
      const int n0 = n_tile * a.block_n;
      const int ab = a.acc_bufs == 2 ? (it & 1) : 0;
      const uint32_t aph = (uint32_t)(a.acc_bufs == 2 ? (it >> 1) : it) & 1u;
      int w0 = 0, h0 = 0, bb = 0;
      uint8_t* stg = sOut + (a.n_sbuf > 1 ? (it % a.n_sbuf) : 0) * n_boxes * TILE_BYTES;

      if (n_tile != cur_n_tile) {   // (re)stage the bias slice of this N tile
        named_bar_sync(2, 128);     // nobody is still reading the old slice
        for (int i = et; i < a.block_n; i += 128) sBias[i] = (a.bias && n0 + i < a.Cout) ? a.bias[n0 + i] : 0.f;
        cur_n_tile = n_tile;
        named_bar_sync(2, 128);
      }
      mbar_wait(&acc_full[ab], aph, 3);
      tc_fence_after();

      for (int j = 0; j < MPAIR; ++j) {
      {
        long long mt = (tile / a.n_tiles) * MPAIR + j;
        w0 = (int)(mt % a.tiles_w) * a.BW; mt /= a.tiles_w;
        h0 = (int)(mt % a.tiles_h) * a.BH;
        bb = (int)(mt / a.tiles_h);
      }
      const bool row_ok = r < rows && (h0 + hl) < a.H && (w0 + wl) < a.W && bb < a.B;
      const long long pix = ((long long)bb * a.H + (h0 + hl)) * a.W + (w0 + wl);
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((ab * MPAIR + j) * a.block_n);
      const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(a.res) + pix * a.Cout + n0;
      __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(a.y) + pix * a.Cout + n0;

      // software pipeline over 16-column chunks: the TMEM load of chunk c+1 is in flight while chunk c
      // is converted and stored
      auto process = [&](const uint32_t (&vv)[16], const int c0) {
        float f[16];
#pragma unroll
        for (int i = 0; i < 16; i += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(sBias + c0 + i);
          f[i] = fminf(fmaxf(__uint_as_float(vv[i]) + b4.x, act_lo), act_hi);
          f[i + 1] = fminf(fmaxf(__uint_as_float(vv[i + 1]) + b4.y, act_lo), act_hi);
          f[i + 2] = fminf(fmaxf(__uint_as_float(vv[i + 2]) + b4.z, act_lo), act_hi);
          f[i + 3] = fminf(fmaxf(__uint_as_float(vv[i + 3]) + b4.w, act_lo), act_hi);
        }
        const bool c_ok0 = n0 + c0 < a.Cout, c_ok1 = n0 + c0 + 8 < a.Cout;   // Cout % 8 == 0
        if (a.res != nullptr && row_ok && c_ok0) {
          uint32_t t[8];
          if (vec32) {
            asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=r"(t[0]), "=r"(t[1]), "=r"(t[2]), "=r"(t[3]), "=r"(t[4]), "=r"(t[5]), "=r"(t[6]), "=r"(t[7])
                         : "l"(rp + c0));
          } else {
            const uint4 u0 = __ldg(reinterpret_cast<const uint4*>(rp + c0));
            uint4 u1 = make_uint4(0, 0, 0, 0);
            if (c_ok1) u1 = __ldg(reinterpret_cast<const uint4*>(rp + c0 + 8));
            t[0] = u0.x; t[1] = u0.y; t[2] = u0.z; t[3] = u0.w; t[4] = u1.x; t[5] = u1.y; t[6] = u1.z; t[7] = u1.w;
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) { f[2 * i] += bf16lo(t[i]); f[2 * i + 1] += bf16hi(t[i]); }
        }
        uint32_t o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = pack_bf16x2(f[2 * i], f[2 * i + 1]);
        if (a.tma_store) {
          const int bx = c0 >> 6, j = (c0 & 63) >> 3;
          uint8_t* rowp = stg + bx * TILE_BYTES + r * 128;
          *reinterpret_cast<uint4*>(rowp + ((j ^ (r & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
          *reinterpret_cast<uint4*>(rowp + (((j + 1) ^ (r & 7)) << 4)) = make_uint4(o[4], o[5], o[6], o[7]);
        } else if (row_ok && c_ok0) {
          if (vec32) {
            asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(yp + c0), "r"(o[0]), "r"(o[1]),
                         "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7])
                         : "memory");
          } else {
            *reinterpret_cast<uint4*>(yp + c0) = make_uint4(o[0], o[1], o[2], o[3]);
            if (c_ok1) *reinterpret_cast<uint4*>(yp + c0 + 8) = make_uint4(o[4], o[5], o[6], o[7]);
          }
        }
      };
      uint32_t va[16], vb[16];
      tmem_ld16(trow, va);
      const int nch = a.block_n >> 4;
      for (int ch = 0; ch < nch; ch += 2) {
        tmem_ld_wait();
        if (ch + 1 < nch) tmem_ld16(trow + (uint32_t)((ch + 1) << 4), vb);
        process(va, ch << 4);
        if (ch + 1 < nch) {
          tmem_ld_wait();
          if (ch + 2 < nch) tmem_ld16(trow + (uint32_t)((ch + 2) << 4), va);
          process(vb, (ch + 1) << 4);
        }
      }
      }   // paired M tiles
      // accumulators fully read -> hand them back to the MMA warp
      tc_fence_before();
      mbar_arrive(&acc_empty[ab]);
      if (a.tma_store) {
        fence_proxy_async_smem();
        // allow n_sbuf-2 stores in flight: the buffer the NEXT tile writes was last read by store(it+1-n_sbuf)
        if (et == 0) {
          if (a.n_sbuf >= 4) asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");
          else if (a.n_sbuf == 3) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          else if (a.n_sbuf == 2) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        named_bar_sync(1, 128);
        if (et == 0) {
          for (int bx = 0; bx < n_boxes; ++bx)
            if (n0 + bx * 64 < a.Cout) tma_store_4d(&tmC, stg + bx * TILE_BYTES, n0 + bx * 64, w0, h0, bb);
          tma_store_commit();
          if (a.n_sbuf == 1) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
        if (a.n_sbuf == 1) named_bar_sync(1, 128);
      }
    }
    if (a.tma_store && et == 0) tma_store_wait_all();
    tc_fence_before();
  }
  if (!a.pdl_early) pdl_trigger();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)a.tmem_cols);
  }
}

static void pick_tile(int W, int H, int* BW, int* BH) {
  // maximise the fraction of the 128 accumulator rows that hold real pixels
  double best = -1.0;
  int bw_best = 1, bh_best = 1;
  const int wmax = W < 128 ? W : 128;
  for (int bw = wmax; bw >= 1; --bw) {
    int bh = 128 / bw;
    if (bh > H) bh = H;
    if (bh < 1) bh = 1;
    const long long tiles = (long long)((W + bw - 1) / bw) * ((H + bh - 1) / bh);
    const double eff = (double)W * H / ((double)tiles * 128.0);
    if (eff > best + 1e-9) { best = eff; bw_best = bw; bh_best = bh; }
    if (bw <= 8 && best > 0) break;
  }
  *BW = bw_best; *BH = bh_best;
}

}  // namespace b200

using namespace b200;

// flags: bit0 epilogue through smem staging + TMA store instead of direct 256-bit register stores;
//        bit1 forbid HALO addressing; bit2 forbid resident weights; bit3 single staging buffer;
//        bit4 HALO descriptors WITH base_offset (experiment: wrong on B200);
//        bits 8..15: force grid size = value * 4 CTAs (0 = auto); bits 16..19: pipeline stages wanted (0 = auto);
//        bits 20..21: CTAs per SM (0 = auto); bit5: never pair M tiles over a shared B stage
// x: [B,H,W,Cin] input; output [B,Ho,Wo,Cout] with Ho = (H-1)/stride+1.  dwmode: w is the block-diagonal
// packing bf16 [C][9][64] (see b200seg_dwconv3x3_tc).  skip (Cs > 0, stride 1, not dwmode): the input is
// cat([skip [B,H,W,Cs], x [B,H,W,Cin-Cs]], channel) and w stays [Cout][taps][Cin].  Issued k-steps per tap set
// equal those of the concatenated input, e.g. the MobileNetV2UNet decoder (Cs + Cu): up1 64 + 1280 -> 84,
// up2 32 + 256 -> 18, up3 24 + 128 -> 10, up4 16 + 64 -> 5 (conv_rs).
static int launch_conv_tc(const void* skip, int Cs, const void* x, const void* w, const float* bias, const void* res,
                          void* y, int B, int H, int W, int Cin, int Cout, int taps, int stride, int dwmode, int act,
                          int flags, cudaStream_t stream) {
  const int Cu = Cin - Cs;
  const int Ho = (H - 1) / stride + 1, Wo = (W - 1) / stride + 1;
  ConvTcArgs a;
  a.bias = bias; a.res = res; a.y = y;
  a.taps = taps; a.Cin = Cin; a.Cout = Cout;
  a.dw = dwmode; a.stride = stride;
  a.halo = (taps == 9 && stride == 1 && W >= 96 && !(flags & 2)) ? 1 : 0;
  if (taps == 1) {   // pointwise: pixels are one flat axis
    const long long M = (long long)B * H * W;
    B200_REQUIRE(M < (1ll << 31), "conv_tc: too many pixels");
    a.W = (int)M; a.H = 1; a.B = 1;
  } else {
    a.W = Wo; a.H = Ho; a.B = B;
  }
  if (a.halo) { a.BW = Wo < 128 ? Wo : 128; a.BH = 1; }
  else pick_tile(a.W, a.H, &a.BW, &a.BH);
  a.tiles_w = (a.W + a.BW - 1) / a.BW;
  a.tiles_h = (a.H + a.BH - 1) / a.BH;
  if (dwmode) {
    // one N tile per 64-channel chunk; its single K chunk is the same 64 input channels
    a.block_n = Cout >= 64 ? 64 : ((Cout + 15) & ~15);
    a.n_tiles = (Cout + 63) / 64;
    a.k_chunks = 1;
  } else {
    // N tiling: one tile if Cout <= 256 (rounded to the UMMA granule 16); otherwise tiles that are a
    // multiple of 64 wide so that a 64-channel store box never spills into a neighbour tile.
    if (Cout <= 256) {
      a.block_n = (Cout + 15) & ~15; a.n_tiles = 1;
    } else {
      int nt = (Cout + 255) / 256;
      int bn = (((Cout + nt - 1) / nt) + 63) & ~63;
      a.block_n = bn; a.n_tiles = (Cout + bn - 1) / bn;
    }
    a.k_chunks = (Cs + 63) / 64 + (Cu + 63) / 64;
  }
  a.Cs = Cs; a.ks = (Cs + 63) / 64;
  a.act = act;
  a.tma_store = flags & 1;
  a.halo_bo = (flags & 16) ? 1 : 0;   // measured on B200: the swizzle uses absolute smem address bits, base_offset must stay 0
  a.tmem_cols = 32;
  while (a.tmem_cols < 2 * a.block_n) a.tmem_cols <<= 1;   // two accumulators

  const int n_boxes = (a.block_n + 63) / 64;
  const int b_tile = a.block_n * 128;
  const int smem_cap = 227 * 1024 - 1024 /*align slack*/ - 1024 /*bias*/ - 256 /*barriers*/;
  a.a_stage_bytes = a.halo ? HALO_BYTES : TILE_BYTES;
  const int kb_per_tile = a.halo ? a.k_chunks * 3 : a.k_chunks * taps;
  const int b_all = taps * a.k_chunks * b_tile;
  a.n_sbuf = 0;
  if (a.tma_store) {
    a.n_sbuf = (flags & 8) ? 1 : 3;
    while (a.n_sbuf > 1 && a.n_sbuf * n_boxes * TILE_BYTES > 64 * 1024) --a.n_sbuf;
  }
  const int out_bytes = a.n_sbuf * n_boxes * TILE_BYTES;
  a.b_resident = (a.n_tiles == 1 && !(flags & 4) && b_all <= 80 * 1024 && b_all + out_bytes + 2 * a.a_stage_bytes <= smem_cap) ? 1 : 0;
  a.b_stage_bytes = a.b_resident ? 0 : (a.halo ? 3 * b_tile : b_tile);
  // streamed weights are the L2->SM bottleneck of the 3x3 layers with large Cin: let two M tiles share every B
  // stage (A traffic unchanged, B traffic halved).  flags bit5 disables.
  a.m_tiles = (long long)a.tiles_w * a.tiles_h * a.B;
  a.mpair = (!a.b_resident && taps * a.k_chunks >= 27 && !a.tma_store && !(flags & 32) && a.m_tiles >= 2) ? 2 : 1;   // measured: pays from ~27 k-blocks
  a.acc_bufs = (a.mpair == 1 || a.block_n <= 64) ? 2 : 1;   // 2 x mpair x block_n columns must fit 512 (and leave room for a 2nd CTA when small)
  a.tmem_cols = 32;
  while (a.tmem_cols < a.acc_bufs * a.mpair * a.block_n) a.tmem_cols <<= 1;
  const int per_stage = a.mpair * a.a_stage_bytes + a.b_stage_bytes;
  const int fixed = out_bytes + (a.b_resident ? b_all : 0);
  // Measured on B200 (tools/kbench.py KB_SWEEP): two resident CTAs per SM (two MMA issuers, two epilogues)
  // beat one CTA with a deeper ring whenever both fit, so: the deepest ring (<= want) that still leaves room
  // for a second CTA (smem and 512 TMEM columns), else the deepest ring that fits at all.
  int want = kb_per_tile <= 3 ? 4 : 6;
  if ((flags >> 16) & 0xf) want = (flags >> 16) & 0xf;
  int stages = (smem_cap - fixed) / per_stage;
  if (stages > want) stages = want;
  if (stages > 8) stages = 8;
  if (!((flags >> 16) & 0xf) && 2 * a.tmem_cols <= 512) {
    const int half_cap = (227 * 1024) / 2 - 1024 - (1024 + 1024 + 256);
    int st2 = (half_cap - fixed) / per_stage;
    if (st2 > want) st2 = want;
    if (st2 >= 2) stages = st2;
  }
  B200_REQUIRE(stages >= 1, "conv_tc: tile does not fit in shared memory (Cin=%d Cout=%d taps=%d)", Cin, Cout, taps);
  a.stages = stages;
  const int smem = fixed + stages * per_stage + 1024 + 1024 + 256;
  B200_REQUIRE(smem <= 227 * 1024, "conv_tc: smem %d too large", smem);
  a.total_tiles = ((a.m_tiles + a.mpair - 1) / a.mpair) * a.n_tiles;

  CUtensorMap tmA, tmB, tmC, tmS;
  {
    // the activation maps always describe the INPUT tensors (U, and S when there is a skip); for 1x1 the pixels
    // are one flat axis
    const uint64_t iw = taps == 1 ? (uint64_t)a.W : (uint64_t)W, ih = taps == 1 ? 1 : (uint64_t)H, ib = taps == 1 ? 1 : (uint64_t)B;
    uint32_t box[4] = {64, (uint32_t)(a.halo ? 130 : a.BW * stride), (uint32_t)(a.BH * stride), 1};
    uint32_t es[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
    for (int src = 0; src < (Cs ? 2 : 1); ++src) {
      const uint64_t c = (uint64_t)(src ? Cs : Cu);
      uint64_t dims[4] = {c, iw, ih, ib};
      uint64_t str[3] = {c * 2, c * 2 * iw, c * 2 * iw * ih};
      int rc = make_tmap_bf16(src ? &tmS : &tmA, src ? skip : x, 4, dims, str, box, 1, es);
      if (rc) return rc;
    }
    if (!Cs) tmS = tmA;
  }
  {
    uint64_t dims[3] = {(uint64_t)(dwmode ? 64 : Cin), (uint64_t)taps, (uint64_t)Cout};
    uint64_t str[2] = {dims[0] * 2, dims[0] * 2 * taps};
    uint32_t box[3] = {64, 1, (uint32_t)a.block_n};
    int rc = make_tmap_bf16(&tmB, w, 3, dims, str, box, 1, nullptr);
    if (rc) return rc;
  }
  {
    uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)a.W, (uint64_t)a.H, (uint64_t)a.B};
    uint64_t str[3] = {(uint64_t)Cout * 2, (uint64_t)Cout * 2 * a.W, (uint64_t)Cout * 2 * a.W * a.H};
    uint32_t box[4] = {64, (uint32_t)a.BW, (uint32_t)a.BH, 1};
    int rc = make_tmap_bf16(&tmC, y, 4, dims, str, box, 1, nullptr);
    if (rc) return rc;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  static bool attr_set[64] = {false};
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_tc_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return set_error((int)e, "conv_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set[dev] = true;
  }
  // persistent grid: as many CTAs as fit (smem and TMEM: 512 columns per SM)
  int per_sm = (227 * 1024) / (smem + 1024);
  if (per_sm > 512 / a.tmem_cols) per_sm = 512 / a.tmem_cols;
  if (per_sm > 2) per_sm = 2;
  if ((flags >> 20) & 0x3) per_sm = (flags >> 20) & 0x3;
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)sm_count() * per_sm;
  if ((flags >> 8) & 0xff) grid = (long long)((flags >> 8) & 0xff) * 4;
  if (grid > a.total_tiles) grid = a.total_tiles;
  a.pdl_early = pdl_mode() != 3;
  auto* kern = a.mpair == 2 ? (Cs ? conv_tc_kernel<2, true> : conv_tc_kernel<2, false>)
                            : (Cs ? conv_tc_kernel<1, true> : conv_tc_kernel<1, false>);
  launch_pdl_if(pdl_mode() > 0, kern, dim3((unsigned)grid), dim3(TC_THREADS), (size_t)smem, stream, tmA, tmB, tmC, tmS, a);
  return check_launch("conv_tc");
}

extern "C" int b200seg_conv_tc(const void* x, const void* w, const float* bias, const void* res, void* y, int B,
                               int H, int W, int Cin, int Cout, int taps, int act, int flags,
                               b200seg_stream_t s) {
  B200_REQUIRE(taps == 1 || taps == 9, "conv_tc: taps=%d (1 or 9)", taps);
  B200_REQUIRE(Cin > 0 && Cin % 8 == 0, "conv_tc: Cin=%d must be a positive multiple of 8", Cin);
  B200_REQUIRE(Cout > 0 && Cout % 8 == 0, "conv_tc: Cout=%d must be a positive multiple of 8", Cout);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "conv_tc: empty tensor");
  B200_REQUIRE(x && w && y, "conv_tc: null pointer");
  return launch_conv_tc(nullptr, 0, x, w, bias, res, y, B, H, W, Cin, Cout, taps, 1, 0, act, flags, (cudaStream_t)s);
}

extern "C" int b200seg_conv_tc_cat(const void* skip, const void* x, const void* w, const float* bias, const void* res,
                                   void* y, int B, int H, int W, int Cs, int Cu, int Cout, int taps, int act, int flags,
                                   b200seg_stream_t s) {
  B200_REQUIRE(taps == 1 || taps == 9, "conv_tc_cat: taps=%d (1 or 9)", taps);
  B200_REQUIRE(Cs >= 0 && Cs % 8 == 0 && Cu > 0 && Cu % 8 == 0, "conv_tc_cat: Cs=%d Cu=%d must be multiples of 8 (Cu > 0)", Cs, Cu);
  B200_REQUIRE(Cout > 0 && Cout % 8 == 0, "conv_tc_cat: Cout=%d must be a positive multiple of 8", Cout);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "conv_tc_cat: empty tensor");
  B200_REQUIRE(x && w && y && (skip || !Cs), "conv_tc_cat: null pointer");
  return launch_conv_tc(skip, Cs, x, w, bias, res, y, B, H, W, Cs + Cu, Cout, taps, 1, 0, act, flags, (cudaStream_t)s);
}

extern "C" int b200seg_dwconv3x3_tc(const void* x, const void* wdiag, const float* bias, void* y, int B, int H,
                                    int W, int C, int stride, int act, int flags, b200seg_stream_t s) {
  B200_REQUIRE(C > 0 && C % 8 == 0, "dwconv3x3_tc: C=%d must be a positive multiple of 8", C);
  B200_REQUIRE(stride == 1 || stride == 2, "dwconv3x3_tc: stride=%d", stride);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "dwconv3x3_tc: empty tensor");
  B200_REQUIRE(x && wdiag && y, "dwconv3x3_tc: null pointer");
  return launch_conv_tc(nullptr, 0, x, wdiag, bias, nullptr, y, B, H, W, C, C, 9, stride, 1, act, flags, (cudaStream_t)s);
}
