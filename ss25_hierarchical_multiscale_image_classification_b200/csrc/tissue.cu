// Tissue segmentation of a low-resolution level ("thumbnail") and the tissue-mask patch filter of the tile scan.
//
// Segmentation is the CLAM-style recipe for CAMELYON16 thumbnails, restated from OpenCV 4.13's 8-bit code paths and
// pinned against the installed cv2 by tests/test_tissue_oracle.py (oracle/tissue.py):
//   cv2.cvtColor(RGB2HSV)[..., 1]  ->  cv2.medianBlur(S, k)  ->  cv2.threshold(BINARY | OTSU) or a fixed threshold.
//   k_sat_median  2-D tiles: saturation S = (d * sdiv[v] + 2048) >> 12 of the tile + halo (clamped coordinates, i.e.
//                 replicated borders) into shared memory, k x k median of S, blurred plane + 256-bin histogram
//   k_otsu        one thread: OpenCV's Otsu loop in fp64 with explicit _rn operations (nvcc would contract into FMA)
//   k_binarize    mask = blurred > t ? 255 : 0, t read from device memory
//
// The filter turns a tissue mask at an integer scale m of the tiled level into a per-candidate keep bit:
//   k_tissue_cells  counts of mask pixels > 0 per g x g level-pixel cell, g = gcd(S, P) (g / m mask pixels a side)
//   k_tissue_flags  a candidate's (P / g)^2 cells summed; bit 0 of its flag = count >= min_tissue_pixels
#include <algorithm>
#include <cfloat>

#include "tile_scan_shared.cuh"
#include "umma.cuh"

namespace hipac {

// OpenCV's saturation table for 8-bit RGB2HSV: sdiv[i] = round(255 * 4096 / i) (no entry falls on a .5)
struct SatTable {
  int v[256];
};
static SatTable make_sat_table() {
  SatTable t;
  t.v[0] = 0;
  for (int i = 1; i < 256; i++) t.v[i] = (int)((255 * 4096 + i / 2) / i);
  return t;
}

__device__ __forceinline__ uint32_t sat_u8(uint32_t r, uint32_t g, uint32_t b, const int* sdiv) {
  const uint32_t v = max(r, max(g, b)), d = v - min(r, min(g, b));
  return (d * (uint32_t)sdiv[v] + 2048u) >> 12;
}

// two 16-bit lanes per register: one compare-exchange of a pixel pair is two instructions (VIMNMX.U16x2)
__device__ __forceinline__ uint32_t min16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("min.u16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t max16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.u16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}

// Median of N = 2M+1 packed values by forgetful selection: the buffer a[s, M+2) starts with M+2 values; each step moves
// its minimum to a[s] and its maximum to a[M+1] with compare-exchanges (per lane, so the two lanes stay independent),
// drops both -- neither can be the median, since each is the extreme of M+2 values -- and refills a[M+1] with the next
// unread value.  After M steps a[M] is the median.
template <int N>
__device__ __forceinline__ uint32_t median_forgetful(uint32_t (&a)[N]) {
  constexpr int M = N / 2;
#pragma unroll
  for (int s = 0; s < M; s++) {
#pragma unroll
    for (int i = s + 1; i < M + 2; i++) {
      const uint32_t lo = min16x2(a[s], a[i]);
      a[i] = max16x2(a[s], a[i]);
      a[s] = lo;
    }
#pragma unroll
    for (int i = s + 1; i < M + 1; i++) {
      const uint32_t hi = max16x2(a[i], a[M + 1]);
      a[i] = min16x2(a[i], a[M + 1]);
      a[M + 1] = hi;
    }
    if (s + 1 < M) a[M + 1] = a[M + 2 + s];
  }
  return a[M];
}

constexpr int kSegTileW = 64;                 // output columns per CTA (32 threads x 2 pixels)
constexpr int kSegTileH = 8;                  // output rows per CTA (one warp per row)
constexpr int kSegFront = 4;                  // shared columns left of the tile (>= the largest radius, even)
constexpr int kSegRowU16 = kSegTileW + 2 * kSegFront;

struct SegParams {
  const uint8_t* rgb;
  int H, W;
  int64_t pitch;
  uint8_t* blur;          // [H][blur_pitch]
  int64_t blur_pitch;
  uint32_t* hist;         // [256], zeroed before the launch
  SatTable sdiv;
};

template <int K>
__global__ void __launch_bounds__(256) k_sat_median(const __grid_constant__ SegParams p) {
  constexpr int R = K / 2, ROWS = kSegTileH + 2 * R;
  __shared__ __align__(16) uint16_t s_sat[ROWS * kSegRowU16];
  __shared__ uint32_t s_hist[256];
  __shared__ int s_sdiv[256];
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * kSegTileW, y0 = blockIdx.y * kSegTileH;
  s_hist[tid] = 0;
  s_sdiv[tid] = p.sdiv.v[tid];
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __syncthreads();
  // ---- saturation of the tile and its halo; clamped coordinates replicate the border and never touch pitch padding ----
  for (int e = tid; e < ROWS * kSegRowU16; e += 256) {
    const int r = e / kSegRowU16, c = e - r * kSegRowU16;
    const int yy = min(max(y0 + r - R, 0), p.H - 1), xx = min(max(x0 + c - kSegFront, 0), p.W - 1);
    const uint8_t* px = p.rgb + (int64_t)yy * p.pitch + (int64_t)xx * 3;
    HIPAC_DEV_ASSERT(yy >= 0 && yy < p.H && xx >= 0 && xx < p.W);
    s_sat[e] = (uint16_t)sat_u8(px[0], px[1], px[2], s_sdiv);
  }
  __syncthreads();
  // ---- k x k median of the pixel pair (x, x + 1): window value (dy, dx) of both pixels packed in one word ----
  const int tx = tid & 31, ty = tid >> 5;
  const int x = x0 + 2 * tx, y = y0 + ty;
  if (y < p.H && x < p.W) {
    uint32_t a[K * K];
#pragma unroll
    for (int dy = 0; dy < K; dy++) {
      // words k = 0..4 hold the shared columns (2tx + 2k, 2tx + 2k + 1) = image columns x - 4 + 2k, x - 3 + 2k
      const uint32_t* wp = reinterpret_cast<const uint32_t*>(s_sat + (ty + dy) * kSegRowU16 + 2 * tx);
      uint32_t w[5];
#pragma unroll
      for (int k = 0; k < 5; k++) w[k] = wp[k];
#pragma unroll
      for (int dx = -R; dx <= R; dx++) {
        const int o = kSegFront + dx;
        a[dy * K + dx + R] = (o & 1) ? __byte_perm(w[o >> 1], w[(o >> 1) + 1], 0x5432) : w[o >> 1];
      }
    }
    uint32_t med;
    if constexpr (K == 1) med = a[0];
    else med = median_forgetful<K * K>(a);
    const uint32_t m0 = med & 0xFFu, m1 = med >> 16;
    uint8_t* out = p.blur + (int64_t)y * p.blur_pitch + x;
    out[0] = (uint8_t)m0;
    atomicAdd(&s_hist[m0], 1u);
    if (x + 1 < p.W) {
      out[1] = (uint8_t)m1;
      atomicAdd(&s_hist[m1], 1u);
    }
  }
  __syncthreads();
  if (s_hist[tid]) atomicAdd(&p.hist[tid], s_hist[tid]);
}

// OpenCV getThreshVal_Otsu_8u, step for step in fp64 (threshold < 0), or the caller's threshold.
__global__ void k_otsu(const uint32_t* __restrict__ hist, int64_t n, int threshold, int32_t* __restrict__ t_out) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (threshold >= 0) {
    t_out[0] = threshold;
    return;
  }
  const double scale = __ddiv_rn(1.0, (double)n);
  double mu = 0.0;
  for (int i = 0; i < 256; i++) mu = __dadd_rn(mu, __dmul_rn((double)i, (double)hist[i]));
  mu = __dmul_rn(mu, scale);
  const double eps = (double)FLT_EPSILON, one_m_eps = __dsub_rn(1.0, (double)FLT_EPSILON);
  double q1 = 0.0, mu1 = 0.0, max_sigma = 0.0;
  int t = 0;
  for (int i = 0; i < 256; i++) {
    const double pi = __dmul_rn((double)hist[i], scale);
    mu1 = __dmul_rn(mu1, q1);
    q1 = __dadd_rn(q1, pi);
    const double q2 = __dsub_rn(1.0, q1);
    if (fmin(q1, q2) < eps || fmax(q1, q2) > one_m_eps) continue;
    mu1 = __ddiv_rn(__dadd_rn(mu1, __dmul_rn((double)i, pi)), q1);
    const double mu2 = __ddiv_rn(__dsub_rn(mu, __dmul_rn(q1, mu1)), q2);
    const double d = __dsub_rn(mu1, mu2);
    const double sigma = __dmul_rn(__dmul_rn(__dmul_rn(q1, q2), d), d);
    if (sigma > max_sigma) max_sigma = sigma, t = i;
  }
  t_out[0] = t;
}

__global__ void __launch_bounds__(256) k_binarize(const uint8_t* __restrict__ blur, int64_t blur_pitch, int H, int W,
                                                  const int32_t* __restrict__ t_in, uint8_t* __restrict__ mask, int64_t mask_pitch) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int x = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (x >= W) return;
  const int t = t_in[0];
  for (int y = blockIdx.y; y < H; y += gridDim.y)
    for (int k = 0; k < 4 && x + k < W; k++) {
      HIPAC_DEV_ASSERT(x + k < W && y < H);
      mask[(int64_t)y * mask_pitch + x + k] = blur[(int64_t)y * blur_pitch + x + k] > t ? 255 : 0;
    }
}

// ------------------------------------------------------------------------------------------
// tissue-mask filter of the tile scan
// ------------------------------------------------------------------------------------------
constexpr int kTissueCellCols = 512;   // mask columns per CTA of k_tissue_cells (rounded to whole cells)

__global__ void __launch_bounds__(256) k_tissue_cells(TissueFilter t) {
  __shared__ uint32_t s_cnt[kTissueCellCols];
  const int cw = t.g / t.m;                                  // mask pixels per cell side
  const int per_cta = max(1, kTissueCellCols / cw);          // cells per CTA
  const int cx_first = blockIdx.x * per_cta, cy = t.cy0 + blockIdx.y;
  for (int k = threadIdx.x; k < per_cta; k += 256) s_cnt[k] = 0;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  __syncthreads();
  const int u0 = cy * cw, u1 = min(u0 + cw, t.h);
  const int v0 = cx_first * cw, v1 = min(min(cx_first + per_cta, t.ncx) * cw, t.w);
  for (int u = u0; u < u1; u++) {
    const uint8_t* row = t.mask + (int64_t)u * t.pitch;
    for (int v = v0 + threadIdx.x; v < v1; v += 256) {
      HIPAC_DEV_ASSERT(u >= 0 && u < t.h && v >= 0 && v < t.w);
      if (row[v]) atomicAdd(&s_cnt[(v - v0) / cw], 1u);
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < per_cta && cx_first + k < t.ncx; k += 256) t.cells[(size_t)blockIdx.y * t.ncx + cx_first + k] = s_cnt[k];
}

__global__ void __launch_bounds__(256) k_tissue_flags(ScanParams p, TissueFilter t, uint8_t* __restrict__ flags, int n_cand) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_cand) return;
  const int ix = idx / p.ny, iyl = idx - ix * p.ny;
  const int cxa = ix * (p.S / t.g), cya = (p.iy_begin + iyl) * (p.S / t.g) - t.cy0, n = p.P / t.g;
  uint32_t cnt = 0;
  for (int dy = 0; dy < n; dy++)
    for (int dx = 0; dx < n; dx++) {
      HIPAC_DEV_ASSERT(cya + dy < t.ncy && cxa + dx < t.ncx);
      cnt += t.cells[(size_t)(cya + dy) * t.ncx + cxa + dx];
    }
  flags[idx] = (flags[idx] & ~1) | (cnt >= (uint32_t)t.min_pixels ? 1 : 0);
}

void tissue_cell_grid(int S, int P, int iy_begin, int nx, int ny, int* g, int* cy0, int* ncx, int* ncy) {
  int a = S, b = P;
  while (b) {
    const int r = a % b;
    a = b, b = r;
  }
  *g = a;
  *cy0 = (int)((int64_t)iy_begin * S / a);
  *ncx = (int)(((int64_t)(nx - 1) * S + P) / a);
  *ncy = (int)(((int64_t)(iy_begin + ny - 1) * S + P) / a) - *cy0;
}

int launch_tissue_filter(const ScanParams& p, const TissueFilter& t, uint8_t* flags, int n_cand, cudaStream_t stream) {
  const int per_cta = std::max(1, kTissueCellCols / (t.g / t.m));
  {
    ProfileScope ps("tissue_cells", stream, (double)std::min((int64_t)t.ncy * (t.g / t.m), (int64_t)t.h) * t.w);
    HIPAC_CHECK_CUDA(launch_ex(k_tissue_cells, dim3((t.ncx + per_cta - 1) / per_cta, t.ncy), dim3(256), 0, stream, 1, t));
  }
  count_launch(1);
  {
    ProfileScope ps("tissue_flags", stream, 0.0);
    HIPAC_CHECK_CUDA(launch_ex(k_tissue_flags, dim3((n_cand + 255) / 256), dim3(256), 0, stream, 1, p, t, flags, n_cand));
  }
  count_launch(1);
  return 0;
}

}  // namespace hipac

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace hipac;

static size_t seg_plane_bytes(int H, int W) { return align_up((size_t)H * W, 256); }

extern "C" size_t hipac_tissue_workspace_bytes(int H, int W) {
  if (H <= 0 || W <= 0) {
    set_error("invalid argument: empty image");
    return 0;
  }
  return 256 * 4 + seg_plane_bytes(H, W);   // histogram, blurred plane
}

template <int K>
static int launch_sat_median(const SegParams& sp, cudaStream_t stream) {
  dim3 grid((sp.W + kSegTileW - 1) / kSegTileW, (sp.H + kSegTileH - 1) / kSegTileH);
  ProfileScope ps("sat_median", stream, (double)sp.H * sp.W * 4);
  HIPAC_CHECK_CUDA(launch_ex(k_sat_median<K>, grid, dim3(256), 0, stream, 1, sp));
  count_launch(1);
  return 0;
}

extern "C" int hipac_tissue_segment(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, int ksize, int threshold,
                                    uint8_t* d_mask, int64_t mask_pitch, int32_t* d_threshold, uint8_t* d_blur,
                                    int64_t blur_pitch, void* d_workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  HIPAC_REQUIRE(H > 0 && W > 0, "empty image");
  HIPAC_REQUIRE((int64_t)H * W < ((int64_t)1 << 32), "image has 2^32 pixels or more");
  HIPAC_REQUIRE(H <= 65535 * kSegTileH, "image taller than 524280 rows");
  HIPAC_REQUIRE(d_rgb && d_mask && d_threshold && d_workspace, "null pointer");
  HIPAC_REQUIRE(pitch_bytes >= (int64_t)W * 3, "pitch smaller than a row");
  HIPAC_REQUIRE(mask_pitch >= W, "mask pitch smaller than a row");
  HIPAC_REQUIRE(!d_blur || blur_pitch >= W, "blur pitch smaller than a row");
  HIPAC_REQUIRE(ksize == 1 || ksize == 3 || ksize == 5 || ksize == 7, "ksize must be 1, 3, 5 or 7");
  HIPAC_REQUIRE(threshold >= -1 && threshold <= 255, "threshold must be -1 (Otsu) or in [0, 255]");
  HIPAC_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "workspace must be 256-byte aligned");
  HIPAC_REQUIRE(workspace_bytes >= hipac_tissue_workspace_bytes(H, W), "workspace too small");
  static const SatTable sdiv = make_sat_table();
  SegParams sp;
  sp.rgb = d_rgb, sp.H = H, sp.W = W, sp.pitch = pitch_bytes, sp.sdiv = sdiv;
  sp.hist = reinterpret_cast<uint32_t*>(d_workspace);
  sp.blur = d_blur ? d_blur : reinterpret_cast<uint8_t*>(d_workspace) + 256 * 4;
  sp.blur_pitch = d_blur ? blur_pitch : W;
  HIPAC_CHECK_CUDA(cudaMemsetAsync(sp.hist, 0, 256 * 4, stream));
  int e = ksize == 1 ? launch_sat_median<1>(sp, stream)
        : ksize == 3 ? launch_sat_median<3>(sp, stream)
        : ksize == 5 ? launch_sat_median<5>(sp, stream)
                     : launch_sat_median<7>(sp, stream);
  if (e) return e;
  {
    ProfileScope ps("otsu", stream, 0.0);
    HIPAC_CHECK_CUDA(launch_ex(k_otsu, dim3(1), dim3(32), 0, stream, 1, (const uint32_t*)sp.hist, (int64_t)H * W, threshold, d_threshold));
  }
  count_launch(1);
  {
    ProfileScope ps("binarize", stream, (double)H * W * 2);
    HIPAC_CHECK_CUDA(launch_ex(k_binarize, dim3((W + 1023) / 1024, std::min(H, 65535)), dim3(256), 0, stream, 1, (const uint8_t*)sp.blur, sp.blur_pitch, H,
                               W, (const int32_t*)d_threshold, d_mask, mask_pitch));
  }
  count_launch(1);
  return 0;
}
