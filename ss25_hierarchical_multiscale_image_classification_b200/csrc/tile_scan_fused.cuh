// Read-once ("fused") stage-1 path.  Included by tile_scan.cu inside namespace hipac (shares its
// __constant__ tables and helpers).
//
// With stride S a multiple of the scale f = P/224, every patch origin lies on the global f-grid, so the
// Pillow-resampled patch equals a 224x224 crop of ONE globally resampled level image D -- except its
// outer ring (output row/column 0 and 223), where Pillow clamps the filter window at the PATCH edge
// (3f/2 taps, renormalised) instead of using the 2f-tap interior window (SURVEY.md section 7, hard part 2).
// Ring rows/columns of all patches fall on a fixed sub-lattice of D (rows k*S/f and k*S/f+223), so the
// streaming pass also emits those rows/columns with the clamped coefficient sets ("variant planes").
//
//   k_cell_stats        one pass over the image (+mask): byte sums / lesion votes per g x g cell, g = gcd(S,P)
//   k_patch_flags       patch sum = sum of its (P/g)^2 cells + white padding -> keep flag + label
//   k_compact           (shared with the direct path) stable compaction in emission order
//   k_downsample_planes one pass over the image: D and its 8 ring-variant planes (skipped when f == 1)
//   k_gather            per survivor: 224x224 crop of the planes -> uint8 / normalised bf16 batch
//
// White padding: pixels right of / below the image read as 255 everywhere (the reference pastes partial
// regions on a white canvas, src/main.py:700-703), which is consistent across all patches because patches
// only ever extend past the right / bottom image edge.
#pragma once

struct FusedGeom {
  int f, lf, Sf, g;        // scale, log2(scale), stride in D pixels, cell size
  int ncx, cy0, ncy;       // cell grid: columns, first stored cell row (global index), stored rows
  int Jbase, Dh, Dw;       // stored D rows [Jbase, Jbase+Dh) and columns [0, Dw)
  int iy_begin, nx, ny;    // candidate grid of this call
  uint32_t* cell_sum;      // [ncy][ncx]
  uint32_t* cell_any;      // [ncy][ncx]
  uint8_t* plane[3][3];    // [vkind][hkind], kinds: 0 interior, 1 top/left clamp, 2 bottom/right clamp
  const uint8_t *ws_lo, *ws_hi;   // the workspace range the planes live in (incl. the tail pad): bounds of every plane read
};

static inline int gcd_int(int a, int b) {
  while (b) {
    int t = a % b;
    a = b, b = t;
  }
  return a;
}

// D-columns per CTA band and D-rows per CTA of k_downsample_planes: a 512 x 224 pixel image tile.
__host__ __device__ constexpr int plane_ci(int f) { return 512 / f; }
__host__ __device__ constexpr int plane_rj(int f) { return 224 / f; }
__host__ __device__ constexpr int plane_ipt(int f) { return f == 8 ? 1 : (f == 4 ? 2 : 4); }

static bool fused_geometry(const ScanParams& p, FusedGeom* G) {
  const int f = p.P / OUT;
  if (p.S % f) return false;
  G->f = f, G->lf = f == 1 ? 0 : (f == 2 ? 1 : (f == 4 ? 2 : 3)), G->Sf = p.S / f;
  G->g = gcd_int(p.S, p.P);
  if (G->g % 32) return false;
  G->iy_begin = p.iy_begin, G->nx = p.nx, G->ny = p.ny;
  G->ncx = (p.W + G->g - 1) / G->g;
  const int ncy_all = (p.H + G->g - 1) / G->g;
  G->cy0 = (int)((int64_t)p.iy_begin * p.S / G->g);
  int cy1 = (int)(((int64_t)(p.iy_begin + p.ny - 1) * p.S + p.P) / G->g);
  if (cy1 > ncy_all) cy1 = ncy_all;
  G->ncy = cy1 > G->cy0 ? cy1 - G->cy0 : 0;
  G->Jbase = p.iy_begin * G->Sf;
  const int jend = (p.iy_begin + p.ny - 1) * G->Sf + OUT;
  const int jimg = (p.H + f / 2 + f - 1) / f;
  G->Dh = (jend < jimg ? jend : jimg) - G->Jbase;
  const int iend = (p.nx - 1) * G->Sf + OUT;
  const int iimg = (p.W + f / 2 + f - 1) / f;
  G->Dw = iend < iimg ? iend : iimg;
  if (f > 1) {
    // every CTA column band must fit its interior + ring-variant columns in 256 * ipt work items
    const int ci = plane_ci(f);
    const int variants = 2 * (ci / G->Sf + 2);
    if ((ci + variants) * 3 > 256 * plane_ipt(f)) return false;
  }
  return G->ncy > 0 && G->Dh > 0 && G->Dw > 0;
}

static size_t fused_plane_bytes(const FusedGeom& G, int v, int h) {
  const size_t rows = v == 0 ? (size_t)G.Dh : (size_t)G.ny;
  const size_t cols = h == 0 ? (size_t)G.Dw : (size_t)G.nx;
  return align_up(rows * cols * 3, 256);
}

static size_t fused_workspace_bytes_impl(const ScanParams& p) {
  FusedGeom G;
  if (!fused_geometry(p, &G)) return 0;
  size_t b = 2 * align_up((size_t)G.ncx * G.ncy * 4, 256);
  if (G.f > 1)
    for (int v = 0; v < 3; v++)
      for (int h = 0; h < 3; h++) b += fused_plane_bytes(G, v, h);
  return b;
}

// ------------------------------------------------------------------------------------------
// pass A1: per-cell byte sums and lesion votes (32-row bands, one warp per row)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_cell_stats(ScanParams p, FusedGeom G, int do_rgb) {
  const int cx = blockIdx.x;
  const int r0 = G.cy0 * G.g + blockIdx.y * 32;
  if (r0 >= p.H) return;
  const int cyl = r0 / G.g - G.cy0;
  const int r1 = min(min(r0 + 32, p.H), (G.cy0 + G.ncy) * G.g);
  const int xb = cx * G.g, xe = min(p.W, xb + G.g);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t s = 0, any = 0;
  const int nbytes = do_rgb ? (xe - xb) * 3 : 0;
  if (!do_rgb) {
  } else if ((p.pitch & 15) == 0 && ((reinterpret_cast<uintptr_t>(p.rgb) + (size_t)xb * 3) & 15) == 0) {
    // fast path: every row of the band starts 16-byte aligned -> flatten (row, chunk) over the CTA and keep
    // several independent 128-bit loads in flight per thread
    const int nfull = nbytes >> 4, nrows = r1 - r0, total = nrows * nfull;
    const uint8_t* base = p.rgb + (int64_t)r0 * p.pitch + (int64_t)xb * 3;
    for (int i0 = threadIdx.x; i0 < total; i0 += 256 * 4) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int idx = i0 + u * 256;
        const int rr = idx / nfull, k = idx - rr * nfull;
        v[u] = idx < total ? ldg_nc_v4(base + (int64_t)rr * p.pitch + k * 16) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 4; u++) s += bytesum4(v[u].x) + bytesum4(v[u].y) + bytesum4(v[u].z) + bytesum4(v[u].w);
    }
    const int tail = nbytes & 15;   // right image edge only
    if (tail)
      for (int idx = threadIdx.x; idx < nrows * tail; idx += 256) s += base[(int64_t)(idx / tail) * p.pitch + nfull * 16 + idx % tail];
  } else {
    for (int r = r0 + warp; r < r1; r += 8)
      s += warp_bytes_sum(p.rgb, (int64_t)r * p.pitch + (int64_t)xb * 3, nbytes, 0, lane);
  }
  if (p.mask) {
    const int mbytes = xe - xb;
    if ((p.mask_pitch & 15) == 0 && ((reinterpret_cast<uintptr_t>(p.mask) + (size_t)xb) & 15) == 0 && (mbytes & 15) == 0) {
      const int nfull = mbytes >> 4, total = (r1 - r0) * nfull;
      const uint8_t* base = p.mask + (int64_t)r0 * p.mask_pitch + xb;
      for (int idx = threadIdx.x; idx < total; idx += 256) {
        const int rr = idx / nfull, k = idx - rr * nfull;
        const uint4 v = ldg_nc_v4(base + (int64_t)rr * p.mask_pitch + k * 16);
        any |= v.x | v.y | v.z | v.w;
      }
    } else {
      for (int r = r0 + warp; r < r1; r += 8) any |= warp_bytes_any(p.mask, (int64_t)r * p.mask_pitch + xb, mbytes, lane);
    }
  }
  for (int o = 16; o; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    any |= __shfl_xor_sync(0xffffffffu, any, o);
  }
  __shared__ uint32_t sh_s[8], sh_a[8];
  if (lane == 0) sh_s[warp] = s, sh_a[warp] = any;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0, a = 0;
    for (int w = 0; w < 8; w++) tot += sh_s[w], a |= sh_a[w];
    if (tot) atomicAdd(&G.cell_sum[(size_t)cyl * G.ncx + cx], tot);  // cell total <= 1792^2*3*255 < 2^32
    if (a) atomicOr(&G.cell_any[(size_t)cyl * G.ncx + cx], 1u);
  }
}

// pass A1': lesion votes only (the streaming pass already produced the byte sums).  The mask is almost everywhere
// zero, so this is a pure stream: every thread ORs 16-byte chunks (4 independent loads in flight) and only a non-zero
// chunk touches its cell (cells are multiples of 32 pixels wide, so an aligned 16-byte chunk never straddles two).
__global__ void __launch_bounds__(256) k_cell_votes(ScanParams p, FusedGeom G, int row0, int nrows) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int cpr = (p.W + 15) >> 4;                       // 16-byte chunks per row (the last one may be partial)
  const int64_t total = (int64_t)nrows * cpr;
  const int64_t step = (int64_t)gridDim.x * 256;
  for (int64_t i0 = (int64_t)blockIdx.x * 256 + threadIdx.x; i0 < total; i0 += 4 * step) {
    uint4 v[4];
    int rr[4], kk[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int64_t i = i0 + u * step;
      v[u] = make_uint4(0, 0, 0, 0);
      rr[u] = 0, kk[u] = 0;
      if (i < total) {
        rr[u] = (int)(i / cpr), kk[u] = (int)(i - (int64_t)rr[u] * cpr);
        const uint8_t* src = p.mask + (int64_t)(row0 + rr[u]) * p.mask_pitch + kk[u] * 16;
        if (kk[u] * 16 + 16 <= p.W) {
          v[u] = ldg_nc_v4(src);
        } else {                                          // ragged right edge: never read the pitch padding
          uint32_t a = 0;
          for (int b = 0; kk[u] * 16 + b < p.W; b++) a |= src[b];
          v[u].x = a;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      if (v[u].x | v[u].y | v[u].z | v[u].w) {
        const int cyl = (row0 + rr[u]) / G.g - G.cy0, cx = kk[u] * 16 / G.g;
        atomicOr(&G.cell_any[(size_t)cyl * G.ncx + cx], 1u);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// per-candidate flags from the cell grid
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_patch_flags(ScanParams p, FusedGeom G, uint8_t* __restrict__ flags, int n_cand) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_cand) return;
  const int ix = idx / p.ny, iyl = idx - ix * p.ny;
  const int x = ix * p.S, y = (p.iy_begin + iyl) * p.S;
  const int pw = min(p.P, p.W - x), ph = min(p.P, p.H - y);
  const int cxa = x / G.g, cya = y / G.g - G.cy0, n = p.P / G.g;
  unsigned long long tot = 0;
  uint32_t a = 0;
  for (int dy = 0; dy < n && cya + dy < G.ncy; dy++)
    for (int dx = 0; dx < n && cxa + dx < G.ncx; dx++) {
      tot += G.cell_sum[(size_t)(cya + dy) * G.ncx + cxa + dx];
      a |= G.cell_any[(size_t)(cya + dy) * G.ncx + cxa + dx];
    }
  tot += 255ull * 3ull * ((unsigned long long)p.P * p.P - (unsigned long long)pw * ph);
  const unsigned long long limit = 240ull * 3ull * (unsigned long long)p.P * p.P;
  flags[idx] = (tot <= limit ? 1 : 0) | (a ? 2 : 0);
}

// ------------------------------------------------------------------------------------------
// pass A2: globally resampled level D + ring-variant planes
//   CTA = 512 x 224 image pixels (+ f-pixel halo) -> (512/f) x (224/f) D pixels.  Image rows stream
//   through a 3-stage cp.async ring of 8 rows; each thread owns up to IPT (column, channel) items and
//   keeps the vertical accumulators of the two D rows an image row contributes to in registers.
// ------------------------------------------------------------------------------------------
constexpr int kPlaneG = 8;        // image rows per pipeline stage
constexpr int kPlaneStages = 3;
constexpr int kPlaneFront = 16;   // front pad so (unused) taps left of pixel 0 stay inside the buffer

__host__ __device__ constexpr int plane_rowcap(int f) { return ((512 + f) * 3 + kPlaneFront + 16 + 16 + 15) / 16 * 16; }

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int F>
__global__ void __launch_bounds__(256) k_downsample_planes(ScanParams p, FusedGeom G) {
  constexpr int CI = plane_ci(F), RJ = plane_rj(F), IPT = plane_ipt(F), ROWCAP = plane_rowcap(F);
  constexpr int NI = 2 * F, NE = 3 * F / 2, HALF = F / 2;
  constexpr int SHIFT = F == 8 ? 7 : (F == 4 ? 5 : 3);  // interior weights are (2m+1) / 2^SHIFT exactly
  constexpr int CH = ROWCAP / 16;                        // 16-byte chunks per staged row (upper bound)
  static_assert(kPlaneG == 8 && 8 % F == 0, "stage rows must be a multiple of the scale");
  extern __shared__ __align__(16) uint8_t sm[];
  uint8_t* rows = sm;                                                       // [stages][G][ROWCAP]
  int* col_I = reinterpret_cast<int*>(sm + kPlaneStages * kPlaneG * ROWCAP);  // D column of each work column
  int* col_kind = col_I + (CI + 2 * (CI / 4 + 2));                          // 0 interior, 1 left, 2 right
  constexpr int HB = 256 * IPT;                                             // bytes per row of the uint8 intermediate
  uint8_t* hbuf = reinterpret_cast<uint8_t*>(col_kind + (CI + 2 * (CI / 4 + 2)));   // [G][HB]
  __shared__ int s_ncols;

  const int I0 = blockIdx.x * CI;
  const int Ja0 = G.Jbase + blockIdx.y * RJ;                // first D row owned by this CTA
  const int Ja1 = min(Ja0 + RJ, G.Jbase + G.Dh);
  const int Ib1 = min(I0 + CI, G.Dw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const CoeffSet& cs = c_coef[G.lf];

  // ---- work columns: interior columns of the band, then the ring-variant columns inside it ----
  if (tid == 0) {
    int n = 0;
    for (int I = I0; I < Ib1; I++) col_I[n] = I, col_kind[n++] = 0;
    for (int I = I0; I < Ib1; I++) {
      if (I % G.Sf == 0 && I / G.Sf < G.nx) col_I[n] = I, col_kind[n++] = 1;
      if (I >= OUT - 1 && (I - (OUT - 1)) % G.Sf == 0 && (I - (OUT - 1)) / G.Sf < G.nx) col_I[n] = I, col_kind[n++] = 2;
    }
    s_ncols = n;
  }
  __syncthreads();
  const int ncols = s_ncols;
  const int n_int = Ib1 - I0;                              // interior columns come first in the work-column table
  const int nitems = ncols * 3;

  // ---- image window of this CTA ----
  const int rfirst = F * Ja0 - HALF;                       // may be < 0 for the first band (rows unused)
  const int rlast = F * Ja1 + HALF;                        // exclusive
  const int px0 = F * I0 - HALF;                           // leftmost pixel any tap may touch
  const int px0c = max(px0, 0);
  const int px1c = min(p.W, F * Ib1 + HALF);               // exclusive, clamped to the image
  const int px1 = F * Ib1 + HALF;
  const int nbytes = (px1c - px0c) * 3;
  const int64_t img_bytes = (int64_t)p.H * p.pitch;
  const int nstage_total = (rlast - rfirst + kPlaneG - 1) / kPlaneG;
  // alignment phase of row r inside its first 16-byte chunk, in 32-bit arithmetic: (r*pitch + px0c*3) mod 16
  const int pm = (int)(p.pitch & 15), pc = (px0c * 3) & 15;
  const uint8_t* col0 = p.rgb + (int64_t)px0c * 3;
  const bool edge_cols = px1 > px1c;

  auto issue_stage = [&](int st) {
    uint8_t* dst_stage = rows + (st % kPlaneStages) * kPlaneG * ROWCAP;
    const int r0 = rfirst + st * kPlaneG;
    for (int idx = tid; idx < kPlaneG * CH; idx += 256) {
      const int rr = idx / CH, k = idx - rr * CH;
      const int r = r0 + rr;
      if (r < 0 || r >= p.H || r >= rlast) continue;
      const int phase = (r * pm + pc) & 15;
      if (k * 16 >= phase + nbytes) continue;
      const uint8_t* src = col0 + (int64_t)r * p.pitch - phase + k * 16;   // 16-byte aligned
      uint8_t* dst = dst_stage + rr * ROWCAP + kPlaneFront + k * 16;         // dst byte b <-> row byte b - phase
      if (src + 16 <= p.rgb + img_bytes) {
        cp_async_16(dst, src);
      } else {
        for (int b = 0; b < 16 && src + b < p.rgb + img_bytes; b++) dst[b] = src[b];
      }
    }
    cp_async_commit();
  };

  // ---- per-item constants and state (items are fixed for the lifetime of the CTA) ----
  int A_int[IPT], A_top[IPT], A_bot[IPT], B_int[IPT], B_top[IPT], B_bot[IPT];
  int it_off[IPT];        // col*3 + c inside hbuf, or -1
  uint8_t* out_int[IPT];  // plane[0][hk] + ccol*3 + c  (row stride it_cw*3)
  uint8_t* out_top[IPT];
  uint8_t* out_bot[IPT];
  int it_cw3[IPT];
#pragma unroll
  for (int q = 0; q < IPT; q++) {
    A_int[q] = A_top[q] = A_bot[q] = B_int[q] = B_top[q] = B_bot[q] = 0;
    const int e = tid + q * 256;
    it_off[q] = -1, out_int[q] = out_top[q] = out_bot[q] = nullptr, it_cw3[q] = 0;
    if (e < nitems) {
      const int c = e / ncols, col = e - c * ncols;
      const int I = col_I[col], kind = col_kind[col];
      const int ixv = kind == 1 ? I / G.Sf : (kind == 2 ? (I - (OUT - 1)) / G.Sf : 0);
      const size_t ccol = kind == 0 ? (size_t)I : (size_t)ixv;
      it_off[q] = col * 3 + c;
      it_cw3[q] = (kind == 0 ? G.Dw : G.nx) * 3;
      out_int[q] = G.plane[0][kind] + ccol * 3 + c;
      out_top[q] = G.plane[1][kind] + ccol * 3 + c;
      out_bot[q] = G.plane[2][kind] + ccol * 3 + c;
    }
  }
  const int Sf = G.Sf, Jbase = G.Jbase, iy_begin = G.iy_begin, ny = G.ny, Himg = p.H;

  for (int st = 0; st < kPlaneStages - 1 && st < nstage_total; st++) issue_stage(st);
  for (int st = 0; st < nstage_total; st++) {
    if (st + kPlaneStages - 1 < nstage_total) {
      issue_stage(st + kPlaneStages - 1);
      cp_async_wait<kPlaneStages - 1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    uint8_t* stage = rows + (st % kPlaneStages) * kPlaneG * ROWCAP;
    const int r_stage = rfirst + st * kPlaneG;
    const int nrows = min(kPlaneG, rlast - r_stage);
    // white fill: rows outside the image, and pixels right of the image edge (edge CTAs only; CTA-uniform test)
    if (r_stage < 0 || r_stage + nrows > Himg || edge_cols) {
      for (int rr = 0; rr < nrows; rr++) {
        const int r = r_stage + rr;
        uint8_t* rowp = stage + rr * ROWCAP;
        if (r < 0 || r >= Himg) {
          for (int k = tid; k < ROWCAP; k += 256) rowp[k] = 255;
        } else if (edge_cols) {
          const int phase = (r * pm + pc) & 15;
          for (int k = nbytes + tid; k < (px1 - px0c) * 3; k += 256) rowp[kPlaneFront + phase + k] = 255;
        }
      }
      __syncthreads();
    }
    // ---- horizontal pass: warp w <-> stage row w, lanes stride over the work columns, 3 channels per item ----
    if (warp < nrows) {
      const int r = r_stage + warp;
      const uint8_t* rowp = stage + warp * ROWCAP;
      const int phase = (r < 0 || r >= Himg) ? 0 : ((r * pm + pc) & 15);
      uint8_t* hrow = hbuf + warp * HB;
      // interior columns col < n_int are I = I0 + col: window start advances by 3F bytes per column
      const int A0 = kPlaneFront + phase + (F * I0 - HALF - px0c) * 3;     // >= 4: the front pad absorbs I == 0
      for (int col = lane; col < n_int; col += 32) {
        uint8_t* hout = hrow + col * 3;
        // 2F taps x 3 interleaved channels = 6F bytes: word loads, funnel-shift to the window start, PRMT the
        // stride-3 bytes of each channel into one register, dp4a with the (2m+1) weights (exact: the weights are
        // (2m+1)/2^SHIFT, so Pillow's 22-bit fixed point reduces to (T + 2^(SHIFT-1)) >> SHIFT)
        const int A = A0 + 3 * F * col;
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(rowp) + (A >> 2);
        const uint32_t sh = (A & 3) * 8;
        constexpr int NW = 6 * F / 4;
        uint32_t wd[NW + 1];
#pragma unroll
        for (int k = 0; k <= NW; k++) wd[k] = wp[k];
#pragma unroll
        for (int k = 0; k < NW; k++) wd[k] = __funnelshift_r(wd[k], wd[k + 1], sh);
        uint32_t T0 = 0, T1 = 0, T2 = 0;
#pragma unroll
        for (int q = 0; q < NI / 4; q++) {
          uint32_t wt = 0;
#pragma unroll
          for (int jj = 0; jj < 4; jj++) {
            const int t = 4 * q + jj;
            wt |= (uint32_t)(t < F ? 2 * t + 1 : 2 * (NI - 1 - t) + 1) << (8 * jj);
          }
          const uint32_t a = wd[3 * q], b = wd[3 * q + 1], cc = wd[3 * q + 2];
          T0 = __dp4a(__byte_perm(__byte_perm(a, b, 0x0630), cc, 0x5210), wt, T0);
          T1 = __dp4a(__byte_perm(__byte_perm(a, b, 0x0741), cc, 0x6210), wt, T1);
          T2 = __dp4a(__byte_perm(__byte_perm(a, b, 0x0052), cc, 0x7410), wt, T2);
        }
        hout[0] = (uint8_t)((T0 + (1u << (SHIFT - 1))) >> SHIFT);
        hout[1] = (uint8_t)((T1 + (1u << (SHIFT - 1))) >> SHIFT);
        hout[2] = (uint8_t)((T2 + (1u << (SHIFT - 1))) >> SHIFT);
      }
      // ring-variant columns (clamped 3F/2-tap windows, 22-bit weights): a handful per band
      for (int col = n_int + lane; col < ncols; col += 32) {
        const int I = col_I[col], kind = col_kind[col];
        uint8_t* hout = hrow + col * 3;
        const uint8_t* pix = rowp + kPlaneFront + phase + (kind == 1 ? F * I - px0c : F * I - HALF - px0c) * 3;
        const int32_t* kh = kind == 1 ? cs.left : cs.right;
        int a0 = 1 << (kPrecisionBits - 1), a1 = a0, a2 = a0;
#pragma unroll
        for (int t = 0; t < NE; t++) {
          a0 += kh[t] * (int)pix[3 * t], a1 += kh[t] * (int)pix[3 * t + 1], a2 += kh[t] * (int)pix[3 * t + 2];
        }
        hout[0] = (uint8_t)min(max(a0 >> kPrecisionBits, 0), 255);
        hout[1] = (uint8_t)min(max(a1 >> kPrecisionBits, 0), 255);
        hout[2] = (uint8_t)min(max(a2 >> kPrecisionBits, 0), 255);
      }
    }
    __syncthreads();
    // ---- vertical pass.  Stage row rr is image row r_stage + rr with (r + HALF) = F * (Ja0 + (8*st + rr) / F) + rr % F,
    //      so the tap index tb = rr % F is a compile-time constant of the unrolled loop. ----
    const int Jstage = Ja0 + (kPlaneG / F) * st;   // D row whose window starts at stage row 0
    // ring-variant accumulators only matter for D rows on the patch-edge lattice (k*Sf and k*Sf + 223); the rows this
    // stage feeds are Jstage-1 .. Jstage + 8/F - 1 (CTA-uniform test)
    bool var = false;
    for (int J = Jstage - 1; J < Jstage + kPlaneG / F; J++) var |= (J >= 0 && J % Sf == 0) || (J >= OUT - 1 && (J - (OUT - 1)) % Sf == 0);
#pragma unroll
    for (int q = 0; q < IPT; q++) {
      if (it_off[q] < 0) continue;
      const uint8_t* hp = hbuf + it_off[q];
#pragma unroll
      for (int rr = 0; rr < kPlaneG; rr++) {
        if (rr >= nrows) break;
        constexpr int kDummy = 0;
        (void)kDummy;
        const int tb = rr % F;
        const int h = hp[rr * HB];
        B_int[q] += (2 * tb + 1) * h;
        A_int[q] += (2 * (F - 1 - tb) + 1) * h;
        if (var) {
          B_bot[q] += cs.right[tb] * h;
          if (tb < HALF) A_bot[q] += cs.right[tb + F] * h;
          if (tb >= HALF) B_top[q] += cs.left[tb - HALF] * h;
          A_top[q] += cs.left[tb + HALF] * h;
        }
        if (tb == F - 1) {
          const int J = Jstage + rr / F - 1;       // the D row that just received its last tap
          if (J >= Ja0 && J < Ja1) {
            out_int[q][(size_t)(J - Jbase) * it_cw3[q]] = (uint8_t)((A_int[q] + (1 << (SHIFT - 1))) >> SHIFT);
            if (J % Sf == 0) {
              const int iy = J / Sf - iy_begin;
              if (iy >= 0 && iy < ny)
                out_top[q][(size_t)iy * it_cw3[q]] = (uint8_t)min(max((A_top[q] + (1 << (kPrecisionBits - 1))) >> kPrecisionBits, 0), 255);
            }
            if (J >= OUT - 1 && (J - (OUT - 1)) % Sf == 0) {
              const int iy = (J - (OUT - 1)) / Sf - iy_begin;
              if (iy >= 0 && iy < ny)
                out_bot[q][(size_t)iy * it_cw3[q]] = (uint8_t)min(max((A_bot[q] + (1 << (kPrecisionBits - 1))) >> kPrecisionBits, 0), 255);
            }
          }
          A_int[q] = B_int[q], A_top[q] = B_top[q], A_bot[q] = B_bot[q];
          B_int[q] = B_top[q] = B_bot[q] = 0;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
constexpr int kGatherPairs = 8;                 // output row pairs per CTA (112 = 14 * 8)

// pass B: gather the 224 x 224 crop of every survivor from the planes (or the image when f == 1).
//   grid (survivor slot, 14 groups of 8 row pairs), 128 threads.  Thread X < 112 owns output columns 2X, 2X+1: per row
//   it reads its 6 source bytes with three aligned 32-bit loads (a warp covers 192 contiguous bytes; the planes are L2
//   resident), funnel-shifts the alignment away, patches the ring pixels (columns 0 / 223 come from the clamp planes)
//   and the white padding, and writes one 32-byte space-to-depth pixel per row pair.  ToTensor + Normalize is one FFMA
//   per value (c_norm_a/c_norm_b, verified at start-up to reproduce the reference's fp32 div/sub/div chain in every one
//   of the 768 (value, channel) cases after bf16 rounding).  No shared memory, no block barrier.
__device__ __forceinline__ float byte_to_float(uint32_t w, int i) {
  // 0x4B0000bb is the float 2^23 + bb: exact uint8 -> float without an integer-to-float conversion
  return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u + i)) - 8388608.0f;
}
__device__ __forceinline__ uint32_t norm_pack(uint32_t w, int i0, int c0, int i1, int c1) {
  const float lo = fmaf(byte_to_float(w, i0), c_norm_a[c0], c_norm_b[c0]);
  const float hi = fmaf(byte_to_float(w, i1), c_norm_a[c1], c_norm_b[c1]);
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

// one 32-byte space-to-depth pixel with a single 256-bit store (sm_100: STG.256), so every L2 sector is written whole
__device__ __forceinline__ void st_global_256(void* dst, const uint4& lo, const uint4& hi) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w), "r"(hi.x),
               "r"(hi.y), "r"(hi.z), "r"(hi.w)
               : "memory");
}

template <bool F1>
__global__ void __launch_bounds__(128) k_gather(ScanParams p, FusedGeom G, OutParams o, const int32_t* __restrict__ coords,
                                                const int32_t* __restrict__ count, int capacity) {
  const int slot = blockIdx.x, jp0 = blockIdx.y * kGatherPairs;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  if (slot >= min(count[0], capacity)) return;
  HIPAC_DEV_ASSERT(slot < capacity);
  __shared__ uint32_t ring[2 * kGatherPairs][2];   // ring pixels (3 bytes) of the CTA's 16 rows: [row][left, right]
  const int x = coords[2 * slot], y = coords[2 * slot + 1];
  const int X = threadIdx.x;
  const bool s2d = o.batch && o.layout == HIPAC_LAYOUT_S2D16_BF16;
  // ---- per-patch constants: where output row j comes from ----
  const uint8_t* base;          // interior source of output row 0, byte 0 = output column 0
  int64_t stride;               // bytes between consecutive output rows
  int nrows, valid;             // rows [0, nrows) exist in the source; bytes [0, valid) of a row exist
  const uint8_t *top = nullptr, *bot = nullptr;       // rows 0 / 223 of the vertically clamped planes
  bool has_right = false;
  if (F1) {
    base = p.rgb + (int64_t)y * p.pitch + (int64_t)x * 3, stride = p.pitch;
    nrows = min(OUT, p.H - y), valid = min(OUT, p.W - x) * 3;
  } else {
    const int J0 = y / G.f - G.Jbase, I0 = x / G.f, iyl = y / p.S - p.iy_begin;
    const size_t ix = (size_t)(x / p.S);
    base = G.plane[0][0] + ((size_t)J0 * G.Dw + I0) * 3, stride = (int64_t)G.Dw * 3;
    nrows = min(OUT, G.Dh - J0), valid = max(0, min(OUT, G.Dw - I0)) * 3;
    top = G.plane[1][0] + ((size_t)iyl * G.Dw + I0) * 3, bot = G.plane[2][0] + ((size_t)iyl * G.Dw + I0) * 3;
    has_right = I0 + OUT - 1 < G.Dw;                     // else column 223 is white via `valid`
    if (X < 4 * kGatherPairs) {                          // stage the ring pixels of this CTA's rows (clamp planes)
      const int rr = X >> 1, side = X & 1, j = 2 * jp0 + rr;
      uint32_t v = 0x00FFFFFFu;
      if (j < nrows && (side == 0 || has_right)) {
        const int vk = j == 0 ? 1 : (j == OUT - 1 ? 2 : 0);
        const size_t row = vk == 0 ? (size_t)(J0 + j) : (size_t)iyl;
        const uint8_t* q = G.plane[vk][1 + side] + (row * G.nx + ix) * 3;
        HIPAC_DEV_ASSERT(q >= G.ws_lo && q + 3 <= G.ws_hi && ix < (size_t)G.nx && row < (size_t)(vk == 0 ? G.Dh : G.ny));
        v = q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16);
      }
      ring[rr][side] = v;
    }
    __syncthreads();
  }
  // thread -> (row-pair group g, column quad Xq): the thread owns output columns 4Xq .. 4Xq+3 (12 source bytes per row, two
  // 32-byte space-to-depth pixels per row pair) of the row pairs g, g+2, g+4, g+6 of this CTA
  const int g = X >> 6, Xq = X & 63;
  constexpr int NQ = OUT / 4;                    // 56 column quads
  if (Xq >= NQ) {
    // threads 56..58 of each group write the explicit zero columns 0, 1, 114 of the padded space-to-depth rows
    if (s2d && Xq < NQ + 3) {
      const int col = Xq - NQ < 2 ? Xq - NQ : HIPAC_S2D16_WIDTH - 1;
      for (int q = g; q < kGatherPairs; q += 2) {
        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
        st_global_256(o.batch + ((((int64_t)slot * (OUT / 2) + jp0 + q) * HIPAC_S2D16_WIDTH + col) << 4), z, z);
      }
    }
    return;
  }
  // ---- per-thread constants ----
  const int nv = valid - 12 * Xq;               // valid bytes among this thread's 12; the rest is white padding
  uint32_t wm[3];
#pragma unroll
  for (int k = 0; k < 3; k++) wm[k] = nv >= 4 * (k + 1) ? 0u : (nv <= 4 * k ? 0xFFFFFFFFu : 0xFFFFFFFFu << (8 * (nv - 4 * k)));
  // ring merge: quad 0 replaces bytes 0..2 (column 0), quad 55 bytes 9..11 (column 223)
  const bool ringL = !F1 && Xq == 0, ringR = !F1 && Xq == NQ - 1 && has_right;
  const uint8_t* img_end = p.rgb + (int64_t)p.H * p.pitch;
  // 12 bytes of one output row (columns 4Xq .. 4Xq+3) as three words; `a` = address of byte 0
  auto fetch = [&](const uint8_t* a, bool row_ok, int rr, uint32_t (&e)[3]) {
    const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(a) & 3) * 8;
    const uint32_t* aw = reinterpret_cast<const uint32_t*>(a - (sh >> 3));
    uint32_t w[4];
    if (!F1 || reinterpret_cast<const uint8_t*>(aw + 4) <= img_end) {
      if (F1) HIPAC_DEV_ASSERT(reinterpret_cast<const uint8_t*>(aw) >= p.rgb);
      else HIPAC_DEV_ASSERT(reinterpret_cast<const uint8_t*>(aw) >= G.ws_lo && reinterpret_cast<const uint8_t*>(aw + 4) <= G.ws_hi);
#pragma unroll
      for (int k = 0; k < 4; k++) w[k] = __ldg(aw + k);
    } else {                                    // last bytes of the level image: never read past the buffer
#pragma unroll
      for (int k = 0; k < 4; k++) w[k] = 0;
      for (int b = 0; b < 16; b++) {
        const uint8_t* q = reinterpret_cast<const uint8_t*>(aw) + b;
        if (q < img_end) w[b >> 2] |= (uint32_t)*q << (8 * (b & 3));
      }
    }
#pragma unroll
    for (int k = 0; k < 3; k++) e[k] = __funnelshift_r(w[k], w[k + 1], sh) | (row_ok ? wm[k] : 0xFFFFFFFFu);
    if (ringL) e[0] = (e[0] & 0xFF000000u) | ring[rr][0];
    if (ringR) e[2] = (e[2] & 0x000000FFu) | (ring[rr][1] << 8);
  };
  const uint8_t* rowp = base + (int64_t)(2 * (jp0 + g)) * stride + 12 * Xq;   // running pointer: row 2*(jp0+q)
  const uint8_t* safe = base + 12 * Xq;                                        // any readable address for rows below the level
#pragma unroll 2
  for (int q = g; q < kGatherPairs; q += 2, rowp += 4 * stride) {
    const int j0 = 2 * (jp0 + q);
    const bool okA = j0 < nrows, okB = j0 + 1 < nrows;
    const uint8_t* pa = !okA ? safe : ((!F1 && j0 == 0) ? top + 12 * Xq : rowp);
    const uint8_t* pb = !okB ? safe : ((!F1 && j0 + 1 == OUT - 1) ? bot + 12 * Xq : rowp + stride);
    uint32_t e[3], f[3];
    fetch(pa, okA, 2 * q, e);
    fetch(pb, okB, 2 * q + 1, f);
    if (o.batch_u8) {
      uint32_t* d0 = reinterpret_cast<uint32_t*>(o.batch_u8 + (((int64_t)slot * OUT + j0) * OUT + 4 * Xq) * 3);
      uint32_t* d1 = d0 + OUT * 3 / 4;
      d0[0] = e[0], d0[1] = e[1], d0[2] = e[2];
      d1[0] = f[0], d1[1] = f[1], d1[2] = f[2];
    }
    if (!o.batch) continue;
    // s2d channel (dy*2+dx)*3+c = dy*6 + (dx*3+c): the 6 bytes a pixel pair takes from a row are already in channel
    // order R G B R G B; bytes 0..5 of the 12 feed s2d pixel 2Xq, bytes 6..11 pixel 2Xq+1
    uint4 lo0, hi0, lo1, hi1;
    lo0.x = norm_pack(e[0], 0, 0, 1, 1);
    lo0.y = norm_pack(e[0], 2, 2, 3, 0);
    lo0.z = norm_pack(e[1], 0, 1, 1, 2);
    lo0.w = norm_pack(f[0], 0, 0, 1, 1);
    hi0.x = norm_pack(f[0], 2, 2, 3, 0);
    hi0.y = norm_pack(f[1], 0, 1, 1, 2);
    hi0.z = hi0.w = 0u;
    lo1.x = norm_pack(e[1], 2, 0, 3, 1);
    lo1.y = norm_pack(e[2], 0, 2, 1, 0);
    lo1.z = norm_pack(e[2], 2, 1, 3, 2);
    lo1.w = norm_pack(f[1], 2, 0, 3, 1);
    hi1.x = norm_pack(f[2], 0, 2, 1, 0);
    hi1.y = norm_pack(f[2], 2, 1, 3, 2);
    hi1.z = hi1.w = 0u;
    if (s2d) {
      uint16_t* dst = o.batch + ((((int64_t)slot * (OUT / 2) + jp0 + q) * HIPAC_S2D16_WIDTH + 2 * Xq + 2) << 4);
      st_global_256(dst, lo0, hi0);
      st_global_256(dst + 16, lo1, hi1);
    } else {
      uint32_t* d0 = reinterpret_cast<uint32_t*>(o.batch + (((int64_t)slot * OUT + j0) * OUT + 4 * Xq) * 3);
      uint32_t* d1 = d0 + OUT * 3 / 2;
      d0[0] = lo0.x, d0[1] = lo0.y, d0[2] = lo0.z, d0[3] = lo1.x, d0[4] = lo1.y, d0[5] = lo1.z;
      d1[0] = lo0.w, d1[1] = hi0.x, d1[2] = hi0.y, d1[3] = lo1.w, d1[4] = hi1.x, d1[5] = hi1.y;
    }
  }
}

#include "tile_scan_stream.cuh"

// ------------------------------------------------------------------------------------------
// host driver
// ------------------------------------------------------------------------------------------
template <int F>
static int launch_planes(const ScanParams& p, const FusedGeom& G, cudaStream_t stream) {
  constexpr int CI = plane_ci(F), RJ = plane_rj(F);
  const size_t smem = (size_t)kPlaneStages * kPlaneG * plane_rowcap(F) + 2 * (CI + 2 * (CI / 4 + 2)) * sizeof(int) +
                      (size_t)kPlaneG * 256 * plane_ipt(F);
  if (int e = ensure_dyn_smem(k_downsample_planes<F>, (int)smem)) return e;
  dim3 grid((G.Dw + CI - 1) / CI, (G.Dh + RJ - 1) / RJ);
  ProfileScope ps("downsample_planes", stream, (double)p.H * p.W * 3);
  k_downsample_planes<F><<<grid, 256, smem, stream>>>(p, G);
  count_launch(1);
  return 0;
}

// ---- streaming pass (tile_scan_stream.cuh) ----
static bool stream_applicable(const ScanParams& p, const FusedGeom& G) {
  if (G.f == 1) return false;
  if ((p.pitch & 15) || (reinterpret_cast<uintptr_t>(p.rgb) & 15)) return false;
  if (G.Sf < 2) return false;
  const int cols = kStripUnits * (8 / G.f);
  if (2 * ((cols + G.Sf - 1) / G.Sf + 1) > kStreamMaxVar) return false;
  return true;
}

template <int F>
static int launch_scan_planes_f(const ScanParams& p, const FusedGeom& G, cudaStream_t stream) {
  const size_t smem = (size_t)kStreamWarps * kStreamStages * (kStreamRows * kStreamRowBytes + 8);
  int sms = 0;
  if (int e = ensure_dyn_smem(k_scan_planes<F>, (int)smem)) return e;
  if (int e = device_sm_count(&sms)) return e;
  static std::atomic<int> per_sm_cached{0};   // a property of the kernel image and the architecture, equal on every B200
  int per_sm = per_sm_cached.load();
  if (!per_sm) {
    HIPAC_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_scan_planes<F>, kStreamWarps * 32, smem));
    if (per_sm < 1) per_sm = 1;
    per_sm_cached.store(per_sm);
  }
  StreamGeom Z;
  Z.n_strips = (G.Dw + kStripUnits * (8 / F) - 1) / (kStripUnits * (8 / F));
  // one resident wave: every warp slot of the GPU gets at most one (strip, row chunk) item of equal height
  const int slots = sms * per_sm * kStreamWarps;
  Z.n_chunks = slots / Z.n_strips;
  if (Z.n_chunks < 1) Z.n_chunks = 1;
  const int min_rows = 4;   // D rows per item: below this the one-block overlap between chunks dominates
  if (Z.n_chunks > (G.Dh + min_rows - 1) / min_rows) Z.n_chunks = (G.Dh + min_rows - 1) / min_rows;
  Z.srow_lo = G.cy0 * G.g;
  Z.srow_hi = min(p.H, (G.cy0 + G.ncy) * G.g);
  const int items = Z.n_strips * Z.n_chunks;
  ProfileScope ps("scan_planes", stream, (double)p.H * p.W * 3);
  HIPAC_CHECK_CUDA(launch_ex(k_scan_planes<F>, dim3((items + kStreamWarps - 1) / kStreamWarps), dim3(kStreamWarps * 32), smem, stream, 1, p, G, Z));
  count_launch(1);
  return 0;
}

static int launch_scan_planes(const ScanParams& p, const FusedGeom& G, cudaStream_t stream) {
  if (G.f == 2) return launch_scan_planes_f<2>(p, G, stream);
  if (G.f == 4) return launch_scan_planes_f<4>(p, G, stream);
  return launch_scan_planes_f<8>(p, G, stream);
}

static int fused_scan_impl(const ScanParams& p, const OutParams& o, uint8_t* flags, int32_t* src_idx, int32_t* block_tot, int32_t* d_coords,
                           uint8_t* d_labels, int32_t* d_count, int capacity, uint8_t* ws, cudaStream_t stream, int keep_all,
                           bool allow_stream, const TissueFilter* tissue, const RoiFilter* roi) {
  FusedGeom G;
  if (!fused_geometry(p, &G)) {
    set_error("fused scan not applicable to this stride / patch size");
    return -4;
  }
  const size_t cell_bytes = align_up((size_t)G.ncx * G.ncy * 4, 256);
  G.cell_sum = reinterpret_cast<uint32_t*>(ws);
  G.cell_any = reinterpret_cast<uint32_t*>(ws + cell_bytes);
  ws += 2 * cell_bytes;
  G.ws_lo = ws;
  for (int v = 0; v < 3; v++)
    for (int h = 0; h < 3; h++) {
      G.plane[v][h] = G.f > 1 ? ws : nullptr;
      if (G.f > 1) ws += fused_plane_bytes(G, v, h);
    }
  G.ws_hi = ws + 1024;   // the tail pad hipac_tile_scan_workspace_bytes adds (the gather reads whole aligned words)
  const int n_cand = p.nx * p.ny;
  HIPAC_CHECK_CUDA(cudaMemsetAsync(G.cell_sum, 0, 2 * cell_bytes, stream));
  const bool stream_ok = allow_stream && stream_applicable(p, G);
  if (stream_ok) {
    // one read of the image: cell sums + resampled planes; the lesion votes come from a mask-only pass
    if (int e = launch_scan_planes(p, G, stream)) return e;
  }
  const int cell_rows = min(p.H, (G.cy0 + G.ncy) * G.g) - G.cy0 * G.g;
  if (stream_ok && p.mask && (p.mask_pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(p.mask) & 15) == 0) {
    const int64_t chunks = (int64_t)cell_rows * ((p.W + 15) >> 4);
    const int64_t want = (chunks + 1023) / 1024;
    const int grid = (int)(want < 148 * 16 ? want : 148 * 16);
    ProfileScope ps("cell_votes", stream, (double)cell_rows * p.W);
    HIPAC_CHECK_CUDA(launch_ex(k_cell_votes, dim3(grid), dim3(256), 0, stream, 1, p, G, G.cy0 * G.g, cell_rows));
    count_launch(1);
  } else if (!stream_ok || p.mask) {
    dim3 grid(G.ncx, (cell_rows + 31) / 32);
    ProfileScope ps(stream_ok ? "cell_votes" : "cell_stats", stream, (double)cell_rows * p.W * ((p.mask ? 1 : 0) + (stream_ok ? 0 : 3)));
    k_cell_stats<<<grid, 256, 0, stream>>>(p, G, stream_ok ? 0 : 1);
    count_launch(1);
  }
  {
    ProfileScope ps("patch_flags", stream, 0.0);
    HIPAC_CHECK_CUDA(launch_ex(k_patch_flags, dim3((n_cand + 255) / 256), dim3(256), 0, stream, 1, p, G, flags, n_cand));
  }
  count_launch(1);
  if (tissue)
    if (int e = launch_tissue_filter(p, *tissue, flags, n_cand, stream)) return e;
  if (roi)
    if (int e = launch_roi_filter(p, *roi, flags, n_cand, stream)) return e;
  if (int e = launch_compact(p, flags, n_cand, d_coords, d_labels, src_idx, d_count, capacity, keep_all, block_tot, stream)) return e;
  if (int e = publish_count(d_count, stream)) return e;
  if ((o.batch_u8 || o.batch) && capacity > 0) {
    if (stream_ok) {
      // planes already written by the streaming pass
    } else if (G.f == 2) {
      if (int e = launch_planes<2>(p, G, stream)) return e;
    } else if (G.f == 4) {
      if (int e = launch_planes<4>(p, G, stream)) return e;
    } else if (G.f == 8) {
      if (int e = launch_planes<8>(p, G, stream)) return e;
    }
    dim3 grid((unsigned)min(n_cand, capacity), OUT / 2 / kGatherPairs);
    ProfileScope ps("gather", stream, 0.0);
    if (G.f == 1) HIPAC_CHECK_CUDA(launch_ex(k_gather<true>, grid, dim3(128), 0, stream, 1, p, G, o, (const int32_t*)d_coords, (const int32_t*)d_count, capacity));
    else HIPAC_CHECK_CUDA(launch_ex(k_gather<false>, grid, dim3(128), 0, stream, 1, p, G, o, (const int32_t*)d_coords, (const int32_t*)d_count, capacity));
    count_launch(1);
  }
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
