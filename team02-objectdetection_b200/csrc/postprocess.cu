// postprocess.cu -- object boxes from the class mask and the colour overlay (inference.py:48-146, overlay_predictions):
//   cv2.resize(mask, (W, H), INTER_NEAREST) -> per selected class: cv2.morphologyEx(plane, MORPH_CLOSE, ones(k, k)) ->
//   cv2.connectedComponentsWithStats(plane, connectivity=8) -> rows (class, label, box, area, centroid)
//   cv2.addWeighted(frame, alpha, palette[resized mask], beta, gamma)
// Each primitive restates the host library's arithmetic, so every value is bit-equal to cv2 4.13:
//   nearest   sx = min(floor(dx * (1.0 / (W / Wm))), Wm - 1) in double, rows alike
//   close     dilate then erode with a k x k rectangle; out-of-image neighbours are ignored (0 for the dilate, 1 for the erode)
//   labels    cv2's default 8-way algorithm (Spaghetti / BBDT) numbers components in the raster order of their first 2x2
//             block (block row y/2, then block column x/2), not of their first pixel.  A union-find over 2x2 blocks whose
//             unions always link the larger root under the smaller index (Allegretti et al. 2019, "BKE") ends with every
//             component rooted at its first block, whatever order the threads ran in; the cv2 label is then 1 + the number
//             of roots before it in its plane.
//   stats     left, top, width, height, area (int32); centroid = (double)sum / area with exact 64-bit coordinate sums
//   blend     saturate(rint_half_even(fmaf(frame, alpha, fmaf(colour, beta, gamma)))) in f32
//
// Kernel sequence of b200seg_detect_objects (one frame = B index, one plane = one frame x one selected class):
//   close_init   resize + membership + all K closes in one pass (one uint16 per pixel, bit i = classes[i]; the dilate is an
//                OR and the erode an AND over the window, separable); writes the closed bitmask and parent[blk] = blk for
//                every foreground 2x2 block of every plane
//   ccl_merge    union with the left, up-left, up and up-right blocks where foreground pixels are 8-adjacent
//   ccl_compress parent[blk] = root; per (plane, 256-block tile) root counts
//   ccl_tiles    one CTA per frame: exclusive scan of the tile counts in plane-major order -> tile offsets, plane bases,
//                component count
//   ccl_number   component id (frame-local, plane-major, cv2 label order) of every root; its statistics slot initialised
//   ccl_stats    per-block partial statistics, aggregated per warp (__match_any_sync on the component) before the atomics
//   ccl_rows     one CTA per frame: scan of area >= min_area -> output rows, count, zeroed rows past the count
//   ccl_labels   (optional) the cv2 label image of every plane, a gather through the root
// Only foreground blocks ever have their parent / id entries written or read (the bitmask decides which blocks those are),
// so the workspace is sized for the worst case but touched in proportion to the objects.
#include "common.cuh"

namespace b200 {

namespace {

constexpr int kTile = 32;              // close_init: 32 x 32 output pixels = 16 x 16 blocks per CTA
constexpr int kRMax = 7;               // k <= 15
constexpr int kReg = kTile + 4 * kRMax; // loaded region: tile + a halo of k - 1 on each side
constexpr int kBlkThreads = 256;       // per-block kernels: one thread = one 2x2 block, a CTA = a tile of 256 blocks
constexpr int kFrameThreads = 1024;    // ccl_tiles / ccl_rows: one CTA per frame

struct CompStats {                     // 40 bytes, one per component
  int area, minx, miny, maxx, maxy, pad;
  unsigned long long sx, sy;
};

struct ClassLut { uint16_t bit[256]; };          // mask value -> class bit (0 if not selected)
struct ClassIds { int id[16]; };                 // plane k -> class value

struct Geometry {
  int B, K, H, W, BH, BW, T;          // T = tiles of 256 blocks per plane
  long long nb;                       // blocks per plane
};

__device__ __forceinline__ int nearest_src(int d, double inv_scale, int ssize) {
  return min((int)floor(__dmul_rn((double)d, inv_scale)), ssize - 1);
}

// block-wide exclusive scan of v (blockDim.x a multiple of 32, <= 1024); *total = the sum over the CTA
__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int n = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += n;
  }
  if (lane == 31) warp_sums[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    int w = lane < nw ? warp_sums[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int n = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += n;
    }
    warp_sums[lane] = w;                 // inclusive over warps
  }
  __syncthreads();
  const int res = inc - v + (wid > 0 ? warp_sums[wid - 1] : 0);
  *total = warp_sums[nw - 1];
  __syncthreads();                       // warp_sums may be reused right after
  return res;
}

// OR of the class bits of the (up to 4) in-image pixels of block (by, bx)
__device__ __forceinline__ uint32_t block_bits(const uint16_t* __restrict__ fb, int by, int bx, int H, int W) {
  const int y = 2 * by, x = 2 * bx;
  const bool x1 = x + 1 < W, y1 = y + 1 < H;
  uint32_t v = fb[(long long)y * W + x];
  if (x1) v |= fb[(long long)y * W + x + 1];
  if (y1) {
    v |= fb[(long long)(y + 1) * W + x];
    if (x1) v |= fb[(long long)(y + 1) * W + x + 1];
  }
  return v;
}

// root of p with path halving: every visited entry is pointed at its grandparent.  Only entries that are no longer roots are
// written, and always with an ancestor (a smaller index of the same set), so racing writers stay correct.  Without it a
// uniform row links every block to its left neighbour and each upward union walks a chain as long as the row.
__device__ __forceinline__ int uf_find(int* P, int p) {
  int q = __ldcg(P + p);
  while (q != p) {
    const int r = __ldcg(P + q);
    if (r == q) return q;
    P[p] = r;
    p = r;
    q = __ldcg(P + p);
  }
  return p;
}

// root of p without writes, for after the merge: a halving write there could land after another thread's final
// parent[p] = root and leave p pointing at a non-root
__device__ __forceinline__ int uf_root(const int* P, int p) {
  int q = P[p];
  while (q != p) { p = q; q = P[p]; }
  return p;
}

// union toward the smaller index: the larger root is hooked under the smaller one with a compare-and-swap that only succeeds
// on a root, so every root is the minimum block index of its set at every point in time
__device__ __forceinline__ void uf_union(int* P, int a, int b) {
  while (true) {
    a = uf_find(P, a);
    b = uf_find(P, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    const int old = atomicCAS(P + b, b, a);
    if (old == b) return;
    b = old;                      // b stopped being a root meanwhile: retry from where it points now
  }
}

}  // namespace

// grid (ceil(W/32), ceil(H/32), B), 256 threads
__global__ void __launch_bounds__(256)
close_init_kernel(const uint8_t* __restrict__ mask, int Hm, int Wm, double inv_sx, double inv_sy, ClassLut lut, int r,
                  Geometry g, uint16_t* __restrict__ bits, int* __restrict__ parent) {
  __shared__ uint16_t sa[kReg][kReg + 2];
  __shared__ uint16_t sb[kReg][kReg + 2];
  __shared__ uint16_t slut[256];
  __shared__ int ssx[kReg], ssy[kReg];
  const int H = g.H, W = g.W, b = blockIdx.z;
  const int tx0 = blockIdx.x * kTile, ty0 = blockIdx.y * kTile;
  const int x0 = tx0 - 2 * r, y0 = ty0 - 2 * r, R = kTile + 4 * r;
  const int tid = threadIdx.x;
  slut[tid] = lut.bit[tid];
  if (tid < R) {
    const int xx = x0 + tid, yy = y0 + tid;
    ssx[tid] = (xx >= 0 && xx < W) ? nearest_src(xx, inv_sx, Wm) : -1;
    ssy[tid] = (yy >= 0 && yy < H) ? nearest_src(yy, inv_sy, Hm) : -1;
  }
  __syncthreads();
  // 1. membership bits of the region (out of image: 0, the dilate's ignored border)
  const uint8_t* mb = mask + (long long)b * Hm * Wm;
  for (int i = tid; i < R * R; i += 256) {
    const int y = i / R, x = i - y * R;
    const int sy = ssy[y], sx = ssx[x];
    sa[y][x] = (sy >= 0 && sx >= 0) ? slut[mb[(long long)sy * Wm + sx]] : (uint16_t)0;
  }
  __syncthreads();
  const int d = 2 * r;                   // window extent - 1
  // 2. horizontal dilate: sb[y][x] = OR sa[y][x .. x+2r], x < 32 + 2r
  const int R1 = kTile + 2 * r;
  for (int i = tid; i < R * R1; i += 256) {
    const int y = i / R1, x = i - y * R1;
    uint32_t v = 0;
    for (int j = 0; j <= d; ++j) v |= sa[y][x + j];
    sb[y][x] = (uint16_t)v;
  }
  __syncthreads();
  // 3. vertical dilate -> D at image (y0 + r + y, x0 + r + x); outside the image D = all ones (the erode's ignored border)
  for (int i = tid; i < R1 * R1; i += 256) {
    const int y = i / R1, x = i - y * R1;
    const int iy = y0 + r + y, ix = x0 + r + x;
    uint32_t v = 0;
    for (int j = 0; j <= d; ++j) v |= sb[y + j][x];
    sa[y][x] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? (uint16_t)v : (uint16_t)0xffff;
  }
  __syncthreads();
  // 4. horizontal erode: sb[y][x] = AND sa[y][x .. x+2r], x < 32
  for (int i = tid; i < R1 * kTile; i += 256) {
    const int y = i / kTile, x = i - y * kTile;
    uint32_t v = 0xffff;
    for (int j = 0; j <= d; ++j) v &= sa[y][x + j];
    sb[y][x] = (uint16_t)v;
  }
  __syncthreads();
  // 5. vertical erode -> the closed bits of the tile (kept in sa for the block pass)
  uint16_t* fb = bits + (long long)b * H * W;
  for (int i = tid; i < kTile * kTile; i += 256) {
    const int y = i / kTile, x = i - y * kTile;
    uint32_t v = 0xffff;
    for (int j = 0; j <= d; ++j) v &= sb[y + j][x];
    const int iy = ty0 + y, ix = tx0 + x;
    const bool in = iy < H && ix < W;
    sa[y][x] = in ? (uint16_t)v : (uint16_t)0;
    if (in) fb[(long long)iy * W + ix] = (uint16_t)v;
  }
  __syncthreads();
  // 6. union-find init: parent[blk] = blk for the foreground blocks of every plane (one thread = one of the 16 x 16 blocks)
  const int lby = tid >> 4, lbx = tid & 15;
  const int by = blockIdx.y * (kTile / 2) + lby, bx = blockIdx.x * (kTile / 2) + lbx;
  if (by < g.BH && bx < g.BW) {
    const uint32_t v = sa[2 * lby][2 * lbx] | sa[2 * lby][2 * lbx + 1] | sa[2 * lby + 1][2 * lbx] | sa[2 * lby + 1][2 * lbx + 1];
    const int blk = by * g.BW + bx;
    for (int k = 0; k < g.K; ++k)
      if ((v >> k) & 1u) parent[((long long)b * g.K + k) * g.nb + blk] = blk;
  }
}

// grid (T, B), 256 threads: one thread = one 2x2 block of all K planes
__global__ void __launch_bounds__(kBlkThreads)
ccl_merge_kernel(const uint16_t* __restrict__ bits, Geometry g, int* parent) {
  const int b = blockIdx.y;
  const int blk = blockIdx.x * kBlkThreads + threadIdx.x;
  if (blk >= g.nb) return;
  const int by = blk / g.BW, bx = blk - by * g.BW;
  const int H = g.H, W = g.W;
  const uint16_t* fb = bits + (long long)b * H * W;
  // the 3 x 4 neighbourhood rows 2by-1 .. 2by+1, columns 2bx-1 .. 2bx+2 (out of image: 0)
  uint32_t p[3][4];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int y = 2 * by - 1 + i;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int x = 2 * bx - 1 + j;
      p[i][j] = (y >= 0 && y < H && x >= 0 && x < W) ? (uint32_t)fb[(long long)y * W + x] : 0u;
    }
  }
  const uint32_t own = p[1][1] | p[1][2] | p[2][1] | p[2][2];
  const uint32_t lcol = p[1][1] | p[2][1], trow = p[1][1] | p[1][2];
  const uint32_t nl = lcol & (p[1][0] | p[2][0]);           // left block's right column
  const uint32_t nul = p[1][1] & p[0][0];                    // up-left corner
  const uint32_t nu = trow & (p[0][1] | p[0][2]);            // up block's bottom row
  const uint32_t nur = p[1][2] & p[0][3];                    // up-right corner
  const uint32_t any = own & (nl | nul | nu | nur);
  if (!any) return;
  for (int k = 0; k < g.K; ++k) {
    const uint32_t m = 1u << k;
    if (!(any & m)) continue;
    int* P = parent + ((long long)b * g.K + k) * g.nb;
    if (nl & m) uf_union(P, blk, blk - 1);
    if (nul & m) uf_union(P, blk, blk - g.BW - 1);
    if (nu & m) uf_union(P, blk, blk - g.BW);
    if (nur & m) uf_union(P, blk, blk - g.BW + 1);
  }
}

// grid (T, B): parent[blk] = root; tile_cnt[(b*K + k)*T + tile] = roots of plane (b, k) in this tile
__global__ void __launch_bounds__(kBlkThreads)
ccl_compress_kernel(const uint16_t* __restrict__ bits, Geometry g, int* parent, int* __restrict__ tile_cnt) {
  const int b = blockIdx.y;
  const int blk = blockIdx.x * kBlkThreads + threadIdx.x;
  const bool valid = blk < g.nb;
  uint32_t own = 0;
  if (valid) {
    const int by = blk / g.BW, bx = blk - by * g.BW;
    own = block_bits(bits + (long long)b * g.H * g.W, by, bx, g.H, g.W);
  }
  for (int k = 0; k < g.K; ++k) {
    bool root = false;
    if ((own >> k) & 1u) {
      int* P = parent + ((long long)b * g.K + k) * g.nb;
      const int r = uf_root(P, blk);
      if (r != blk) P[blk] = r;
      root = r == blk;
    }
    const int n = __syncthreads_count(root);
    if (threadIdx.x == 0) tile_cnt[((long long)b * g.K + k) * g.T + blockIdx.x] = n;
  }
}

// grid B, 1024 threads: tile offsets (components before the tile in the frame, plane-major), plane bases, component count
__global__ void __launch_bounds__(kFrameThreads)
ccl_tiles_kernel(Geometry g, const int* __restrict__ tile_cnt, int* __restrict__ tile_off, int* __restrict__ plane_base,
                 int* __restrict__ ncomp) {
  __shared__ int ws[32];
  const int b = blockIdx.x;
  const long long n = (long long)g.K * g.T;
  const int* cnt = tile_cnt + (long long)b * n;
  int* off = tile_off + (long long)b * n;
  int carry = 0;
  for (long long base = 0; base < n; base += kFrameThreads) {
    const long long i = base + threadIdx.x;
    const int v = i < n ? cnt[i] : 0;
    int total;
    const int e = block_exclusive_scan(v, ws, &total);
    if (i < n) {
      off[i] = carry + e;
      if (i % g.T == 0) plane_base[(long long)b * g.K + i / g.T] = carry + e;
    }
    carry += total;
  }
  if (threadIdx.x == 0) ncomp[b] = carry;
}

// grid (T, B): component id of every root (frame-local; its cv2 label is id - plane_base + 1) and its statistics slot
__global__ void __launch_bounds__(kBlkThreads)
ccl_number_kernel(const uint16_t* __restrict__ bits, Geometry g, const int* __restrict__ parent, const int* __restrict__ tile_off,
                  int* __restrict__ cid, CompStats* __restrict__ stats) {
  __shared__ int ws[32];
  const int b = blockIdx.y;
  const int blk = blockIdx.x * kBlkThreads + threadIdx.x;
  const bool valid = blk < g.nb;
  uint32_t own = 0;
  if (valid) {
    const int by = blk / g.BW, bx = blk - by * g.BW;
    own = block_bits(bits + (long long)b * g.H * g.W, by, bx, g.H, g.W);
  }
  const long long cmax = (long long)g.K * g.nb;          // statistics slots per frame
  for (int k = 0; k < g.K; ++k) {
    const long long plane = (long long)b * g.K + k;
    const bool root = ((own >> k) & 1u) && parent[plane * g.nb + blk] == blk;
    int total;
    const int e = block_exclusive_scan(root ? 1 : 0, ws, &total);
    if (root) {
      const int c = tile_off[plane * g.T + blockIdx.x] + e;
      cid[plane * g.nb + blk] = c;
      CompStats s;
      s.area = 0; s.minx = 0x7fffffff; s.miny = 0x7fffffff; s.maxx = -1; s.maxy = -1; s.pad = 0; s.sx = 0; s.sy = 0;
      stats[b * cmax + c] = s;
    }
  }
}

// grid (T, B): area, box and coordinate sums of every component; the lanes of a warp that hit the same component add
// their partials first (__match_any_sync + __reduce_*_sync), so a component that covers half the frame costs one set of
// atomics per warp, not per pixel
__global__ void __launch_bounds__(kBlkThreads)
ccl_stats_kernel(const uint16_t* __restrict__ bits, Geometry g, const int* __restrict__ parent, const int* __restrict__ cid,
                 CompStats* __restrict__ stats) {
  const int b = blockIdx.y;
  const int blk = blockIdx.x * kBlkThreads + threadIdx.x;
  const bool valid = blk < g.nb;
  const int H = g.H, W = g.W;
  int by = 0, bx = 0;
  uint32_t q[4] = {0u, 0u, 0u, 0u};                     // the block's pixels a, b (top row), c, d
  if (valid) {
    by = blk / g.BW; bx = blk - by * g.BW;
    const uint16_t* fb = bits + (long long)b * H * W;
    const int y = 2 * by, x = 2 * bx;
    const bool x1 = x + 1 < W, y1 = y + 1 < H;
    q[0] = fb[(long long)y * W + x];
    if (x1) q[1] = fb[(long long)y * W + x + 1];
    if (y1) q[2] = fb[(long long)(y + 1) * W + x];
    if (x1 && y1) q[3] = fb[(long long)(y + 1) * W + x + 1];
  }
  const uint32_t own = q[0] | q[1] | q[2] | q[3];
  if (__all_sync(0xffffffffu, own == 0)) return;
  const long long cmax = (long long)g.K * g.nb;
  const int lane = threadIdx.x & 31;
  for (int k = 0; k < g.K; ++k) {
    const uint32_t m = 1u << k;
    const bool fg = (own & m) != 0;
    if (!__any_sync(0xffffffffu, fg)) continue;
    unsigned long long key = ~0ull;
    unsigned area = 0, sx = 0, sy = 0;
    int minx = 0x7fffffff, miny = 0x7fffffff, maxx = -1, maxy = -1;
    if (fg) {
      const long long plane = (long long)b * g.K + k;
      const int root = parent[plane * g.nb + blk];
      key = (unsigned long long)(b * cmax + cid[plane * g.nb + root]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (q[j] & m) {
          const int x = 2 * bx + (j & 1), y = 2 * by + (j >> 1);
          ++area; sx += x; sy += y;
          minx = min(minx, x); maxx = max(maxx, x); miny = min(miny, y); maxy = max(maxy, y);
        }
      }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    area = __reduce_add_sync(peers, area);
    sx = __reduce_add_sync(peers, sx);                  // < 128 * W: exact in 32 bits (W <= 2^20)
    sy = __reduce_add_sync(peers, sy);
    minx = __reduce_min_sync(peers, minx);
    miny = __reduce_min_sync(peers, miny);
    maxx = __reduce_max_sync(peers, maxx);
    maxy = __reduce_max_sync(peers, maxy);
    if (fg && (__ffs(peers) - 1) == lane) {
      CompStats* s = stats + key;
      atomicAdd(&s->area, (int)area);
      atomicMin(&s->minx, minx);
      atomicMin(&s->miny, miny);
      atomicMax(&s->maxx, maxx);
      atomicMax(&s->maxy, maxy);
      atomicAdd(&s->sx, (unsigned long long)sx);
      atomicAdd(&s->sy, (unsigned long long)sy);
    }
  }
}

// grid B, 1024 threads: rows of the components with area >= min_area in (class position, label) order
__global__ void __launch_bounds__(kFrameThreads)
ccl_rows_kernel(Geometry g, ClassIds cls, const CompStats* __restrict__ stats, const int* __restrict__ plane_base,
                const int* __restrict__ ncomp, int min_area, int max_objects, int* __restrict__ count, int* __restrict__ out_stats,
                double* __restrict__ out_cent) {
  __shared__ int ws[32];
  __shared__ int pb[16];
  const int b = blockIdx.x;
  if (threadIdx.x < g.K) pb[threadIdx.x] = plane_base[(long long)b * g.K + threadIdx.x];
  __syncthreads();
  const int n = ncomp[b];
  const CompStats* st = stats + (long long)b * g.K * g.nb;
  int* os = out_stats + (long long)b * max_objects * 7;
  double* oc = out_cent + (long long)b * max_objects * 2;
  int carry = 0;
  for (int base = 0; base < n; base += kFrameThreads) {
    const int c = base + threadIdx.x;
    CompStats s;
    bool keep = false;
    if (c < n) {
      s = st[c];
      keep = s.area >= min_area;
    }
    int total;
    const int row = carry + block_exclusive_scan(keep ? 1 : 0, ws, &total);
    if (keep && row < max_objects) {
      int k = 0;
      while (k + 1 < g.K && pb[k + 1] <= c) ++k;
      int* o = os + (long long)row * 7;
      o[0] = cls.id[k];
      o[1] = c - pb[k] + 1;
      o[2] = s.minx;
      o[3] = s.miny;
      o[4] = s.maxx - s.minx + 1;
      o[5] = s.maxy - s.miny + 1;
      o[6] = s.area;
      oc[2 * row] = __ddiv_rn((double)s.sx, (double)s.area);
      oc[2 * row + 1] = __ddiv_rn((double)s.sy, (double)s.area);
    }
    carry += total;
  }
  if (threadIdx.x == 0) count[b] = carry;
  for (int row = min(carry, max_objects) + threadIdx.x; row < max_objects; row += kFrameThreads) {
#pragma unroll
    for (int j = 0; j < 7; ++j) os[(long long)row * 7 + j] = 0;
    oc[2 * row] = 0.0;
    oc[2 * row + 1] = 0.0;
  }
}

// one thread per pixel: labels[b, k, y, x] = cv2 label of the pixel in plane (b, k), 0 for background
__global__ void __launch_bounds__(256)
ccl_labels_kernel(const uint16_t* __restrict__ bits, Geometry g, const int* __restrict__ parent, const int* __restrict__ cid,
                  const int* __restrict__ plane_base, int* __restrict__ labels) {
  const long long HW = (long long)g.H * g.W;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)g.B * HW) return;
  const int b = (int)(i / HW);
  const long long p = i - b * HW;
  const int y = (int)(p / g.W), x = (int)(p - (long long)y * g.W);
  const uint32_t v = bits[i];
  const int blk = (y >> 1) * g.BW + (x >> 1);
  for (int k = 0; k < g.K; ++k) {
    const long long plane = (long long)b * g.K + k;
    int l = 0;
    if ((v >> k) & 1u) l = cid[plane * g.nb + parent[plane * g.nb + blk]] - plane_base[plane] + 1;
    labels[plane * HW + p] = l;
  }
}

// overlay: out = saturate(rint(fmaf(frame, alpha, fmaf(palette[nearest mask], beta, gamma)))), BGR uint8.  VEC = 16: a
// thread blends 16 consecutive pixels with three 16-byte loads and three 16-byte stores; VEC = 1: one pixel, byte access.
template <int VEC>
__global__ void __launch_bounds__(256)
overlay_kernel(const uint8_t* __restrict__ frames, const uint8_t* __restrict__ mask, int Hm, int Wm, int H, int W, double inv_sx,
               double inv_sy, const uint8_t* __restrict__ palette, int npal, float alpha, float beta, float gamma,
               uint8_t* __restrict__ out, long long npix) {
  __shared__ uint32_t pal[256];
  {
    const int t = threadIdx.x;
    pal[t] = t < npal ? (uint32_t)palette[3 * t] | ((uint32_t)palette[3 * t + 1] << 8) | ((uint32_t)palette[3 * t + 2] << 16) : 0u;
  }
  __syncthreads();
  const long long p0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (p0 >= npix) return;
  const long long HW = (long long)H * W;
  int b = (int)(p0 / HW);
  const long long rem = p0 - b * HW;
  int y = (int)(rem / W), x = (int)(rem - (long long)y * W);
  uint8_t f[VEC * 3];
  if (VEC == 16) {
    const uint4* src = reinterpret_cast<const uint4*>(frames + p0 * 3);
#pragma unroll
    for (int q = 0; q < 3; ++q) *reinterpret_cast<uint4*>(f + 16 * q) = __ldg(src + q);
  } else {
#pragma unroll
    for (int j = 0; j < VEC * 3; ++j) f[j] = frames[p0 * 3 + j];
  }
  uint8_t o[VEC * 3];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    const int sy = nearest_src(y, inv_sy, Hm), sx = nearest_src(x, inv_sx, Wm);
    const uint32_t col = pal[mask[((long long)b * Hm + sy) * Wm + sx]];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = __fmaf_rn((float)f[3 * j + c], alpha, __fmaf_rn((float)((col >> (8 * c)) & 255u), beta, gamma));
      o[3 * j + c] = (uint8_t)min(max(__float2int_rn(v), 0), 255);
    }
    if (++x == W) { x = 0; if (++y == H) { y = 0; ++b; } }
  }
  if (VEC == 16) {
    uint4* dst = reinterpret_cast<uint4*>(out + p0 * 3);
#pragma unroll
    for (int q = 0; q < 3; ++q) dst[q] = *reinterpret_cast<const uint4*>(o + 16 * q);
  } else {
#pragma unroll
    for (int j = 0; j < VEC * 3; ++j) out[p0 * 3 + j] = o[j];
  }
}

namespace {

Geometry make_geometry(int B, int K, int H, int W) {
  Geometry g;
  g.B = B; g.K = K; g.H = H; g.W = W;
  g.BH = (H + 1) / 2; g.BW = (W + 1) / 2;
  g.nb = (long long)g.BH * g.BW;
  g.T = (int)((g.nb + kBlkThreads - 1) / kBlkThreads);
  return g;
}

long long align256(long long v) { return (v + 255) & ~255ll; }

// workspace layout: bits u16 [B,H,W] | parent i32 [B,K,nb] | cid i32 [B,K,nb] | stats CompStats [B, K*nb] |
// tile_cnt i32 [B,K,T] | tile_off i32 [B,K,T] | plane_base i32 [B,K] | ncomp i32 [B]
struct Workspace {
  long long bits, parent, cid, stats, tile_cnt, tile_off, plane_base, ncomp, total;
};
Workspace workspace_layout(const Geometry& g) {
  Workspace w;
  const long long planes = (long long)g.B * g.K, blocks = planes * g.nb, tiles = planes * g.T;
  long long o = 0;
  w.bits = o;       o = align256(o + (long long)g.B * g.H * g.W * 2);
  w.parent = o;     o = align256(o + blocks * 4);
  w.cid = o;        o = align256(o + blocks * 4);
  w.stats = o;      o = align256(o + blocks * (long long)sizeof(CompStats));
  w.tile_cnt = o;   o = align256(o + tiles * 4);
  w.tile_off = o;   o = align256(o + tiles * 4);
  w.plane_base = o; o = align256(o + planes * 4);
  w.ncomp = o;      o = align256(o + (long long)g.B * 4);
  w.total = o;
  return w;
}

int check_detect_shape(int B, int K, int H, int W) {
  B200_REQUIRE(K >= 1 && K <= 16, "detect_objects: %d classes (1..16: one bit each in a uint16 per pixel)", K);
  B200_REQUIRE(B > 0 && H > 0 && W > 0, "detect_objects: non-positive size B=%d H=%d W=%d", B, H, W);
  B200_REQUIRE(B <= 65535, "detect_objects: B=%d frames (at most 65535 per call)", B);
  B200_REQUIRE(H <= (1 << 20) && W <= (1 << 20) && (long long)H * W < (1ll << 31),
               "detect_objects: frame %dx%d too large (sides <= 2^20, fewer than 2^31 pixels)", W, H);
  const Geometry g = make_geometry(B, K, H, W);
  B200_REQUIRE((long long)K * g.nb < (1ll << 31), "detect_objects: more than 2^31 component slots per frame");
  return 0;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" int b200seg_detect_workspace_bytes(int B, int K, int H, int W, long long* bytes) {
  B200_REQUIRE(bytes, "detect_workspace_bytes: null pointer");
  const int rc = check_detect_shape(B, K, H, W);
  if (rc) return rc;
  *bytes = workspace_layout(make_geometry(B, K, H, W)).total;
  return 0;
}

extern "C" int b200seg_detect_objects(const uint8_t* mask, int B, int Hm, int Wm, int H, int W, const int* classes, int K,
                                      int close, int min_area, int max_objects, void* workspace, long long workspace_bytes,
                                      int* count, int* stats, double* centroid, int* labels, b200seg_stream_t s) {
  B200_REQUIRE(mask && classes && workspace && count && stats && centroid, "detect_objects: null pointer");
  B200_REQUIRE(Hm > 0 && Wm > 0, "detect_objects: non-positive mask size %dx%d", Wm, Hm);
  const int rc = check_detect_shape(B, K, H, W);
  if (rc) return rc;
  B200_REQUIRE(close >= 1 && close <= 2 * kRMax + 1 && (close & 1), "detect_objects: close=%d (odd, 1..15)", close);
  B200_REQUIRE(max_objects >= 1, "detect_objects: max_objects=%d (>= 1)", max_objects);
  ClassLut lut;
  ClassIds ids;
  for (int i = 0; i < 256; ++i) lut.bit[i] = 0;
  for (int i = 0; i < 16; ++i) ids.id[i] = 0;
  for (int i = 0; i < K; ++i) {
    B200_REQUIRE(classes[i] >= 0 && classes[i] <= 255, "detect_objects: class id %d outside [0, 255]", classes[i]);
    B200_REQUIRE(lut.bit[classes[i]] == 0, "detect_objects: class %d listed twice", classes[i]);
    lut.bit[classes[i]] = (uint16_t)(1u << i);
    ids.id[i] = classes[i];
  }
  const Geometry g = make_geometry(B, K, H, W);
  const Workspace w = workspace_layout(g);
  B200_REQUIRE(workspace_bytes >= w.total, "detect_objects: workspace of %lld bytes, %lld needed", workspace_bytes, w.total);
  B200_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "detect_objects: workspace must be 256-byte aligned");
  char* ws = static_cast<char*>(workspace);
  uint16_t* bits = reinterpret_cast<uint16_t*>(ws + w.bits);
  int* parent = reinterpret_cast<int*>(ws + w.parent);
  int* cid = reinterpret_cast<int*>(ws + w.cid);
  CompStats* cst = reinterpret_cast<CompStats*>(ws + w.stats);
  int* tile_cnt = reinterpret_cast<int*>(ws + w.tile_cnt);
  int* tile_off = reinterpret_cast<int*>(ws + w.tile_off);
  int* plane_base = reinterpret_cast<int*>(ws + w.plane_base);
  int* ncomp = reinterpret_cast<int*>(ws + w.ncomp);
  cudaStream_t st = (cudaStream_t)s;
  // cv2's nearest map: ifx = 1 / (dst / src) in double
  const double inv_sx = 1.0 / ((double)W / (double)Wm), inv_sy = 1.0 / ((double)H / (double)Hm);
  const dim3 gt((W + kTile - 1) / kTile, (H + kTile - 1) / kTile, B);
  close_init_kernel<<<gt, 256, 0, st>>>(mask, Hm, Wm, inv_sx, inv_sy, lut, close / 2, g, bits, parent);
  int e = check_launch("detect_objects: close_init");
  if (e) return e;
  const dim3 gb(g.T, B);
  ccl_merge_kernel<<<gb, kBlkThreads, 0, st>>>(bits, g, parent);
  if ((e = check_launch("detect_objects: ccl_merge"))) return e;
  ccl_compress_kernel<<<gb, kBlkThreads, 0, st>>>(bits, g, parent, tile_cnt);
  if ((e = check_launch("detect_objects: ccl_compress"))) return e;
  ccl_tiles_kernel<<<B, kFrameThreads, 0, st>>>(g, tile_cnt, tile_off, plane_base, ncomp);
  if ((e = check_launch("detect_objects: ccl_tiles"))) return e;
  ccl_number_kernel<<<gb, kBlkThreads, 0, st>>>(bits, g, parent, tile_off, cid, cst);
  if ((e = check_launch("detect_objects: ccl_number"))) return e;
  ccl_stats_kernel<<<gb, kBlkThreads, 0, st>>>(bits, g, parent, cid, cst);
  if ((e = check_launch("detect_objects: ccl_stats"))) return e;
  ccl_rows_kernel<<<B, kFrameThreads, 0, st>>>(g, ids, cst, plane_base, ncomp, min_area, max_objects, count, stats, centroid);
  if ((e = check_launch("detect_objects: ccl_rows"))) return e;
  if (labels) {
    const long long n = (long long)B * H * W;
    B200_REQUIRE((n + 255) / 256 < (1ll << 31), "detect_objects: too many pixels for the label image");
    ccl_labels_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(bits, g, parent, cid, plane_base, labels);
    if ((e = check_launch("detect_objects: ccl_labels"))) return e;
  }
  return 0;
}

extern "C" int b200seg_overlay(const uint8_t* frames, const uint8_t* mask, int B, int Hm, int Wm, int H, int W,
                               const uint8_t* palette, int npal, float alpha, float beta, float gamma, uint8_t* out,
                               b200seg_stream_t s) {
  B200_REQUIRE(frames && mask && out && (palette || npal == 0), "overlay: null pointer");
  B200_REQUIRE(B > 0 && Hm > 0 && Wm > 0 && H > 0 && W > 0, "overlay: non-positive size");
  B200_REQUIRE(npal >= 0 && npal <= 256, "overlay: palette of %d colours (0..256)", npal);
  const long long npix = (long long)B * H * W;
  const double inv_sx = 1.0 / ((double)W / (double)Wm), inv_sy = 1.0 / ((double)H / (double)Hm);
  cudaStream_t st = (cudaStream_t)s;
  if (npix % 16 == 0 && (reinterpret_cast<uintptr_t>(frames) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
    const long long g = (npix / 16 + 255) / 256;
    B200_REQUIRE(g < (1ll << 31), "overlay: too many pixels");
    overlay_kernel<16><<<(unsigned)g, 256, 0, st>>>(frames, mask, Hm, Wm, H, W, inv_sx, inv_sy, palette, npal, alpha, beta,
                                                    gamma, out, npix);
  } else {
    const long long g = (npix + 255) / 256;
    B200_REQUIRE(g < (1ll << 31), "overlay: too many pixels");
    overlay_kernel<1><<<(unsigned)g, 256, 0, st>>>(frames, mask, Hm, Wm, H, W, inv_sx, inv_sy, palette, npal, alpha, beta,
                                                   gamma, out, npix);
  }
  return check_launch("overlay");
}
