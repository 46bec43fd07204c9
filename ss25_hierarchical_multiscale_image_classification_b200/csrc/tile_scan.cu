// Stage 1 of the HiPAC hot path: multiscale patch extraction of one level image in HBM.
// Replaces the hot loop of the reference's extract_patches (src/main.py:682-727) plus the
// Resize/ToTensor/Normalize of its feature-extraction transform (src/main.py:812-818).
// See include/hipac_b200.h for the contract and DESIGN.md for the kernels' rooflines.
#include <atomic>
#include <mutex>

#include "common.cuh"
#include "pillow_coeffs.h"
#include "tile_scan_shared.cuh"
#include "umma.cuh"

namespace hipac {

// ------------------------------------------------------------------------------------------
// constant tables
// ------------------------------------------------------------------------------------------
__constant__ CoeffSet c_coef[4];          // index log2(scale); [0] unused
__constant__ uint16_t c_lut_bf16[768];    // [v][c] -> bf16 bits of (v/255 - mean_c)/std_c
__device__ uint16_t g_lut_bf16[768];      // same table in global memory (gathered with divergent indices)
__constant__ float c_norm_a[3], c_norm_b[3];   // y = fma(v, a_c, b_c): one-instruction form of the table (checked at start-up)

static const float kMean[3] = {0.485f, 0.456f, 0.406f};  // reference src/main.py:816
static const float kStd[3] = {0.229f, 0.224f, 0.225f};

static uint16_t f32_to_bf16_rne(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

void host_normalize_lut_bf16(uint16_t* lut) {
  for (int v = 0; v < 256; v++)
    for (int c = 0; c < 3; c++) {
      volatile float x = (float)v / 255.0f;       // ToTensor: uint8 -> float32 / 255
      volatile float y = (x - kMean[c]) / kStd[c];  // Normalize: sub then div, fp32
      lut[v * 3 + c] = f32_to_bf16_rne(y);
    }
}

// Once per device, under a mutex: the tables are copied on the caller's stream and the stream is synchronised BEFORE the
// device is marked done, and a second thread / stream asking meanwhile blocks on the mutex -- so no launch on any stream
// can read the __constant__ tables before they have landed.
static int upload_constants(cudaStream_t stream) {
  static std::mutex mu;
  static bool done[64] = {};
  int dev = 0;
  HIPAC_CHECK_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (dev < 64 && done[dev]) return 0;
  static CoeffSet h_coef[4];
  static uint16_t h_lut[768];
  for (int l = 1; l <= 3; l++) {
    PillowCoeffs pc = build_pillow_coeffs(1 << l);
    if (!pc.ok) {
      set_error("Pillow coefficient structure check failed");
      return -3;
    }
    for (int t = 0; t < 16; t++) h_coef[l].interior[t] = pc.interior[t];
    for (int t = 0; t < 12; t++) h_coef[l].left[t] = pc.left[t], h_coef[l].right[t] = pc.right[t];
  }
  host_normalize_lut_bf16(h_lut);
  // single-FMA form of ToTensor+Normalize used by the gather kernel; it must reproduce the table bit for bit
  float h_a[3], h_b[3];
  for (int c = 0; c < 3; c++) {
    h_a[c] = (float)(1.0 / (255.0 * (double)kStd[c]));
    h_b[c] = (float)(-(double)kMean[c] / (double)kStd[c]);
    for (int v = 0; v < 256; v++) {
      if (f32_to_bf16_rne(fmaf((float)v, h_a[c], h_b[c])) != h_lut[v * 3 + c]) {
        set_error("single-FMA normalisation does not reproduce the fp32 ToTensor/Normalize table");
        return -3;
      }
    }
  }
  HIPAC_CHECK_CUDA(cudaMemcpyToSymbolAsync(c_norm_a, h_a, sizeof(h_a), 0, cudaMemcpyHostToDevice, stream));
  HIPAC_CHECK_CUDA(cudaMemcpyToSymbolAsync(c_norm_b, h_b, sizeof(h_b), 0, cudaMemcpyHostToDevice, stream));
  HIPAC_CHECK_CUDA(cudaMemcpyToSymbolAsync(c_coef, h_coef, sizeof(h_coef), 0, cudaMemcpyHostToDevice, stream));
  HIPAC_CHECK_CUDA(cudaMemcpyToSymbolAsync(c_lut_bf16, h_lut, sizeof(h_lut), 0, cudaMemcpyHostToDevice, stream));
  HIPAC_CHECK_CUDA(cudaMemcpyToSymbolAsync(g_lut_bf16, h_lut, sizeof(h_lut), 0, cudaMemcpyHostToDevice, stream));
  HIPAC_CHECK_CUDA(cudaStreamSynchronize(stream));
  if (dev < 64) done[dev] = true;
  return 0;
}

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__device__ __forceinline__ uint32_t bytesum4(uint32_t w) { return __vsadu4(w, 0u); }

// Sum of the bytes [start, start+n) of `base`, computed by one warp; `limit` = size of the buffer.
__device__ __forceinline__ uint32_t warp_bytes_sum(const uint8_t* base, int64_t start, int n, int64_t limit, int lane) {
  uint32_t s = 0;
  const int64_t end = start + n;
  for (int64_t a = (start & ~int64_t(15)) + lane * 16; a < end; a += 32 * 16) {
    if (a >= start && a + 16 <= end) {
      uint4 v = ldg_nc_v4(base + a);
      s += bytesum4(v.x) + bytesum4(v.y) + bytesum4(v.z) + bytesum4(v.w);
    } else {
      int64_t lo = a < start ? start : a, hi = a + 16 < end ? a + 16 : end;
      for (int64_t b = lo; b < hi; b++) s += base[b];
    }
  }
  (void)limit;
  return s;
}

__device__ __forceinline__ uint32_t warp_bytes_any(const uint8_t* base, int64_t start, int n, int lane) {
  uint32_t s = 0;
  const int64_t end = start + n;
  for (int64_t a = (start & ~int64_t(15)) + lane * 16; a < end; a += 32 * 16) {
    if (a >= start && a + 16 <= end) {
      uint4 v = ldg_nc_v4(base + a);
      s |= v.x | v.y | v.z | v.w;
    } else {
      int64_t lo = a < start ? start : a, hi = a + 16 < end ? a + 16 : end;
      for (int64_t b = lo; b < hi; b++) s |= base[b];
    }
  }
  return s;
}

// ------------------------------------------------------------------------------------------
// DIRECT path, kernel 1: per-candidate tissue sum + lesion vote (any stride)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_stats_direct(ScanParams p, uint8_t* __restrict__ flags) {
  const int idx = blockIdx.x;
  const int ix = idx / p.ny, iyl = idx - ix * p.ny;
  const int x = ix * p.S, y = (p.iy_begin + iyl) * p.S;
  const int pw = min(p.P, p.W - x), ph = min(p.P, p.H - y);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t s = 0, any = 0;
  for (int r = warp; r < ph; r += 8) {
    s += warp_bytes_sum(p.rgb, (int64_t)(y + r) * p.pitch + (int64_t)x * 3, pw * 3, (int64_t)p.H * p.pitch, lane);
    if (p.mask) any |= warp_bytes_any(p.mask, (int64_t)(y + r) * p.mask_pitch + x, pw, lane);
  }
  __shared__ uint32_t sh_s[8], sh_a[8];
  for (int o = 16; o; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    any |= __shfl_xor_sync(0xffffffffu, any, o);
  }
  if (lane == 0) sh_s[warp] = s, sh_a[warp] = any;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long tot = 0;
    uint32_t a = 0;
    for (int w = 0; w < 8; w++) tot += sh_s[w], a |= sh_a[w];
    tot += 255ull * 3ull * ((unsigned long long)p.P * p.P - (unsigned long long)pw * ph);  // white padding
    const unsigned long long limit = 240ull * 3ull * (unsigned long long)p.P * p.P;        // mean > 240 -> reject
    flags[idx] = (tot <= limit ? 1 : 0) | (a ? 2 : 0);
  }
}

// ------------------------------------------------------------------------------------------
// compaction: stable (emission-order) prefix sum over the candidate flags.
//   Blocks of 1024 candidates.  k_compact_count leaves the survivors per block in block_tot; in k_compact every CTA sums
//   the totals of the blocks before it (a few hundred values even for a 100k x 100k level) and scatters its own block with
//   a ballot/popc scan -- no inter-CTA waiting, any number of candidates.  With one block the count kernel is skipped.
// ------------------------------------------------------------------------------------------
constexpr int kCompactBlock = 1024;

__global__ void __launch_bounds__(kCompactBlock) k_compact_count(const uint8_t* __restrict__ flags, int n_cand, int keep_all,
                                                                int32_t* __restrict__ block_tot) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int idx = blockIdx.x * kCompactBlock + threadIdx.x;
  const int keep = idx < n_cand ? ((flags[idx] & 1) | keep_all) : 0;
  const int n = __syncthreads_count(keep);
  if (threadIdx.x == 0) block_tot[blockIdx.x] = n;
}

__global__ void __launch_bounds__(kCompactBlock) k_compact(ScanParams p, const uint8_t* __restrict__ flags, int n_cand,
                                                          int32_t* __restrict__ coords, uint8_t* __restrict__ labels,
                                                          int32_t* __restrict__ src_idx, int32_t* __restrict__ count,
                                                          int capacity, int keep_all, const int32_t* __restrict__ block_tot) {
  __shared__ int warp_tot[32];
  __shared__ int s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  // ---- survivors in the blocks before this one ----
  int part = 0;
  for (int b = threadIdx.x; b < (int)blockIdx.x; b += kCompactBlock) part += block_tot[b];
  part = __reduce_add_sync(0xffffffffu, part);
  if (lane == 0) warp_tot[warp] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < 32; w++) t += warp_tot[w];
    s_base = t;
  }
  __syncthreads();
  const int base = s_base;
  __syncthreads();
  // ---- this block ----
  const int idx = blockIdx.x * kCompactBlock + threadIdx.x;
  const uint8_t f = idx < n_cand ? flags[idx] : 0;
  const int keep = idx < n_cand ? ((f & 1) | keep_all) : 0;
  const unsigned b = __ballot_sync(0xffffffffu, keep);
  const int pre = __popc(b & ((1u << lane) - 1));
  if (lane == 0) warp_tot[warp] = __popc(b);
  __syncthreads();
  int woff = 0, tot = 0;
  for (int w = 0; w < 32; w++) {
    woff += w < warp ? warp_tot[w] : 0;
    tot += warp_tot[w];
  }
  const int slot = base + woff + pre;
  if (keep && slot < capacity) {
    const int ix = idx / p.ny, iyl = idx - ix * p.ny;
    coords[2 * slot + 0] = ix * p.S;
    coords[2 * slot + 1] = (p.iy_begin + iyl) * p.S;
    labels[slot] = (f >> 1) & 1;
    src_idx[slot] = idx;
  }
  if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
    count[0] = base + tot;
    count[1] = n_cand;
  }
}

// flags -> compacted survivors (one or two launches); block_tot holds one int per 1024 candidates
static int launch_compact(const ScanParams& p, const uint8_t* flags, int n_cand, int32_t* d_coords, uint8_t* d_labels,
                          int32_t* src_idx, int32_t* d_count, int capacity, int keep_all, int32_t* block_tot, cudaStream_t stream) {
  const int nb = (n_cand + kCompactBlock - 1) / kCompactBlock;
  ProfileScope ps("compact", stream, (double)n_cand);
  if (nb > 1) {
    HIPAC_CHECK_CUDA(launch_ex(k_compact_count, dim3(nb), dim3(kCompactBlock), 0, stream, 1, flags, n_cand, keep_all, block_tot));
    count_launch(1);
  }
  HIPAC_CHECK_CUDA(launch_ex(k_compact, dim3(nb), dim3(kCompactBlock), 0, stream, 1, p, flags, n_cand, d_coords, d_labels, src_idx, d_count,
                             capacity, keep_all, (const int32_t*)block_tot));
  count_launch(1);
  return 0;
}

// ------------------------------------------------------------------------------------------
// output writer shared by the direct and fused resamplers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void write_output(const OutParams& o, int slot, int j, int i, int c, uint32_t v) {
  if (o.batch_u8) o.batch_u8[(((int64_t)slot * OUT + j) * OUT + i) * 3 + c] = (uint8_t)v;
  if (o.batch) {
    const uint16_t b = c_lut_bf16[v * 3 + c];
    if (o.layout == HIPAC_LAYOUT_NHWC3_BF16) {
      o.batch[(((int64_t)slot * OUT + j) * OUT + i) * 3 + c] = b;
    } else {
      o.batch[((((int64_t)slot * (OUT / 2) + (j >> 1)) * HIPAC_S2D16_WIDTH + (i >> 1) + 2) << 4) + ((j & 1) * 2 + (i & 1)) * 3 + c] = b;
    }
  }
}

__device__ __forceinline__ void write_s2d_pad(const OutParams& o, int slot, int j) {
  if (o.batch && o.layout == HIPAC_LAYOUT_S2D16_BF16 && (j & 1)) {
    uint16_t* row = o.batch + (((int64_t)slot * (OUT / 2) + (j >> 1)) * HIPAC_S2D16_WIDTH << 4);
    for (int X = threadIdx.x; X < OUT / 2; X += blockDim.x) *reinterpret_cast<uint2*>(row + ((X + 2) << 4) + 12) = make_uint2(0u, 0u);
    if (threadIdx.x < 3) {  // explicit zero columns 0, 1 and 114
      uint4* q = reinterpret_cast<uint4*>(row + ((threadIdx.x < 2 ? threadIdx.x : HIPAC_S2D16_WIDTH - 1) << 4));
      q[0] = q[1] = make_uint4(0u, 0u, 0u, 0u);
    }
  }
}

// ------------------------------------------------------------------------------------------
// DIRECT path, kernel 2: Pillow-exact resample of one surviving patch row (any stride)
//   grid (survivor slot, output row j); horizontal pass of the <=16 input rows of the vertical
//   window into shared memory (uint8 intermediate, as Pillow), then the vertical pass.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_resample_direct(ScanParams p, OutParams o, const int32_t* __restrict__ coords,
                                                         const int32_t* __restrict__ count, int capacity) {
  const int slot = blockIdx.x, j = blockIdx.y;
  const int n = min(count[0], capacity);
  if (slot >= n) return;
  const int x = coords[2 * slot], y = coords[2 * slot + 1];
  const int f = p.P / OUT;
  __shared__ __align__(16) uint8_t rowbuf[1792 * 3 + 32];
  __shared__ uint8_t hbuf[16][OUT * 3];
  const int tid = threadIdx.x;
  const int64_t img_bytes = (int64_t)p.H * p.pitch;

  if (f == 1) {  // PIL resize is the identity when the patch is already 224x224
    const int yy = y + j;
    for (int e = tid; e < OUT * 3; e += 256) {
      const int i = e / 3, c = e - 3 * i;
      uint32_t v = 255;
      if (yy < p.H && x + i < p.W) v = p.rgb[(int64_t)yy * p.pitch + (int64_t)(x + i) * 3 + c];
      write_output(o, slot, j, i, c, v);
    }
    write_s2d_pad(o, slot, j);
    return;
  }

  const int lf = f == 2 ? 1 : (f == 4 ? 2 : 3);
  const CoeffSet& cs = c_coef[lf];
  const int ni = 2 * f, ne = 3 * f / 2;
  // vertical window of output row j
  const int vmin = j == 0 ? 0 : f * j - f / 2;
  const int vcnt = (j == 0 || j == OUT - 1) ? ne : ni;
  const int32_t* kv = j == 0 ? cs.left : (j == OUT - 1 ? cs.right : cs.interior);
  const int pw = min(p.P, p.W - x);

  for (int r = 0; r < vcnt; r++) {
    const int yy = y + vmin + r;
    // ---- stage the patch row (white beyond the image) ----
    const int64_t start = (int64_t)yy * p.pitch + (int64_t)x * 3;
    const int phase = (int)(start & 15);
    uint8_t* rb = rowbuf + phase;  // rb[k] = byte k of the patch row
    if (yy < p.H) {
      const int64_t end = start + (int64_t)pw * 3;
      for (int64_t a = (start & ~int64_t(15)) + tid * 16; a < end; a += 256 * 16) {
        uint8_t* dst = rowbuf + (a - (start & ~int64_t(15)));
        if (a + 16 <= img_bytes) {
          *reinterpret_cast<uint4*>(dst) = ldg_nc_v4(p.rgb + a);
        } else {
          for (int b = 0; b < 16 && a + b < img_bytes; b++) dst[b] = p.rgb[a + b];
        }
      }
      __syncthreads();
      for (int e = pw * 3 + tid; e < p.P * 3; e += 256) rb[e] = 255;
    } else {
      for (int e = tid; e < p.P * 3; e += 256) rb[e] = 255;
    }
    __syncthreads();
    // ---- horizontal pass -> uint8 intermediate ----
    for (int e = tid; e < OUT * 3; e += 256) {
      const int i = e / 3, c = e - 3 * i;
      const int hmin = i == 0 ? 0 : f * i - f / 2;
      const int hcnt = (i == 0 || i == OUT - 1) ? ne : ni;
      const int32_t* kh = i == 0 ? cs.left : (i == OUT - 1 ? cs.right : cs.interior);
      int acc = 1 << (kPrecisionBits - 1);
      for (int t = 0; t < hcnt; t++) acc += kh[t] * (int)rb[(hmin + t) * 3 + c];
      acc >>= kPrecisionBits;
      hbuf[r][e] = (uint8_t)min(max(acc, 0), 255);
    }
    __syncthreads();
  }
  // ---- vertical pass ----
  for (int e = tid; e < OUT * 3; e += 256) {
    const int i = e / 3, c = e - 3 * i;
    int acc = 1 << (kPrecisionBits - 1);
    for (int r = 0; r < vcnt; r++) acc += kv[r] * (int)hbuf[r][e];
    acc >>= kPrecisionBits;
    write_output(o, slot, j, i, c, (uint32_t)min(max(acc, 0), 255));
  }
  write_s2d_pad(o, slot, j);
}

// Early publication of the survivor count: right after the compaction kernel the two counters are copied to a pinned
// host buffer and an event is recorded, so the caller can size the next stage while the (much longer) resample /
// gather kernels of this call are still running.
static thread_local int32_t* g_count_host = nullptr;   // set by hipac_tile_scan_set_count_buffer
static thread_local cudaEvent_t g_count_events[64] = {};   // one per device: an event belongs to the device it was created on
static thread_local cudaEvent_t g_count_event = nullptr;   // the event of this thread's most recent scan

static int publish_count(const int32_t* d_count, cudaStream_t stream) {
  if (!g_count_host) return 0;
  int dev = 0;
  HIPAC_CHECK_CUDA(cudaGetDevice(&dev));
  HIPAC_REQUIRE(dev < 64, "device index above 63");
  if (!g_count_events[dev]) HIPAC_CHECK_CUDA(cudaEventCreateWithFlags(&g_count_events[dev], cudaEventDisableTiming));
  g_count_event = g_count_events[dev];
  HIPAC_CHECK_CUDA(cudaMemcpyAsync(g_count_host, d_count, 8, cudaMemcpyDeviceToHost, stream));
  HIPAC_CHECK_CUDA(cudaEventRecord(g_count_event, stream));
  return 0;
}

#include "tile_scan_fused.cuh"

}  // namespace hipac

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace hipac;

extern "C" int hipac_pillow_coeffs(int scale, int32_t* h_interior, int32_t* h_left, int32_t* h_right) {
  PillowCoeffs pc = build_pillow_coeffs(scale);
  HIPAC_REQUIRE(pc.ok, "scale must be 2, 4 or 8");
  for (int t = 0; t < 2 * scale; t++) h_interior[t] = pc.interior[t];
  for (int t = 0; t < 3 * scale / 2; t++) h_left[t] = pc.left[t], h_right[t] = pc.right[t];
  return 0;
}

extern "C" int hipac_normalize_lut_bf16(uint16_t* h_lut) {
  HIPAC_REQUIRE(h_lut != nullptr, "null lut");
  host_normalize_lut_bf16(h_lut);
  return 0;
}

static int scan_geometry(int H, int W, int P, int S, int iy_begin, int iy_end, int* nx, int* ny) {
  HIPAC_REQUIRE(H > 0 && W > 0, "empty level image");
  HIPAC_REQUIRE(P == 224 || P == 448 || P == 896 || P == 1792, "patch size must be 1792>>level");
  HIPAC_REQUIRE(S > 0, "stride must be positive");
  const int ny_all = (H + S - 1) / S;
  HIPAC_REQUIRE(iy_begin >= 0 && iy_begin <= iy_end && iy_end <= ny_all, "grid row range out of bounds");
  *nx = (W + S - 1) / S;
  *ny = iy_end - iy_begin;
  return 0;
}

extern "C" size_t hipac_tile_scan_workspace_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int mode) {
  mode &= ~(HIPAC_SCAN_KEEP_ALL | HIPAC_SCAN_NO_STREAM);
  int nx, ny;
  if (scan_geometry(H, W, P, S, iy_begin, iy_end, &nx, &ny)) return 0;
  const size_t n_cand = (size_t)nx * ny;
  size_t b = align_up(n_cand, 256) + align_up(n_cand * 4, 256) +                      // flags + src_idx
             align_up(((n_cand + kCompactBlock - 1) / kCompactBlock) * 4, 256);        // survivors per compaction block
  if (mode != HIPAC_SCAN_DIRECT) {
    ScanParams p{};
    p.H = H, p.W = W, p.P = P, p.S = S, p.nx = nx, p.ny = ny, p.iy_begin = iy_begin;
    b += fused_workspace_bytes_impl(p);
  }
  // tail pad: the gather kernel reads whole 32-bit words up to one patch row (224 * 3 bytes) past the end of a plane
  return b + 1024;
}

static int tissue_geometry(int P, int S, int m) {
  HIPAC_REQUIRE(m == 1 || m == 2 || m == 4 || m == 8 || m == 16 || m == 32, "tissue_scale must be a power of two up to 32");
  HIPAC_REQUIRE(S % m == 0 && P % m == 0, "stride and patch size must be multiples of tissue_scale");
  return 0;
}

// bytes of the tissue cell grid, which precedes the hipac_tile_scan workspace layout (0 on error)
static size_t tissue_cell_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int m) {
  int nx, ny;
  if (scan_geometry(H, W, P, S, iy_begin, iy_end, &nx, &ny) || tissue_geometry(P, S, m)) return 0;
  if ((int64_t)nx * ny == 0) return 256;
  int g, cy0, ncx, ncy;
  tissue_cell_grid(S, P, iy_begin, nx, ny, &g, &cy0, &ncx, &ncy);
  return align_up((size_t)ncx * ncy * 4, 256);
}

extern "C" size_t hipac_tile_scan_tissue_workspace_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int mode, int tissue_scale) {
  const size_t cells = tissue_cell_bytes(H, W, P, S, iy_begin, iy_end, tissue_scale);
  const size_t base = cells ? hipac_tile_scan_workspace_bytes(H, W, P, S, iy_begin, iy_end, mode) : 0;
  return base ? cells + base : 0;
}

static int tile_scan_impl(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, const uint8_t* d_mask, int64_t mask_pitch, int P,
                          int S, int iy_begin, int iy_end, int32_t* d_coords, uint8_t* d_labels, uint8_t* d_batch_u8, void* d_batch,
                          int layout, int32_t* d_count, int capacity, void* d_workspace, size_t workspace_bytes, int mode,
                          TissueFilter* tissue, const RoiFilter* roi, cudaStream_t stream) {
  const int keep_all = (mode & HIPAC_SCAN_KEEP_ALL) ? 1 : 0;
  const bool allow_stream = !(mode & HIPAC_SCAN_NO_STREAM);   // HIPAC_SCAN_NO_STREAM: force the cp.async kernels (cross-check)
  mode &= ~(HIPAC_SCAN_KEEP_ALL | HIPAC_SCAN_NO_STREAM);
  int nx, ny;
  if (int e = scan_geometry(H, W, P, S, iy_begin, iy_end, &nx, &ny)) return e;
  HIPAC_REQUIRE(d_rgb && d_coords && d_labels && d_count && d_workspace, "null pointer");
  HIPAC_REQUIRE(pitch_bytes >= (int64_t)W * 3, "pitch smaller than a row");
  HIPAC_REQUIRE(!d_mask || mask_pitch >= W, "mask pitch smaller than a row");
  HIPAC_REQUIRE(capacity >= 0, "negative capacity");
  HIPAC_REQUIRE(!d_batch || layout == HIPAC_LAYOUT_NHWC3_BF16 || layout == HIPAC_LAYOUT_S2D16_BF16, "unknown batch layout");
  HIPAC_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "workspace must be 256-byte aligned");
  HIPAC_REQUIRE(((uintptr_t)d_batch_u8 & 15) == 0 && ((uintptr_t)d_batch & 31) == 0, "batch buffers must be 16/32-byte aligned");
  HIPAC_REQUIRE(workspace_bytes >= hipac_tile_scan_workspace_bytes(H, W, P, S, iy_begin, iy_end, mode), "workspace too small");
  HIPAC_REQUIRE((int64_t)nx * ny < (int64_t)1 << 30, "too many candidates for one call; split the row range");
  HIPAC_REQUIRE(mode == HIPAC_SCAN_AUTO || mode == HIPAC_SCAN_DIRECT || mode == HIPAC_SCAN_FUSED, "unknown scan mode");
  HIPAC_REQUIRE(!(keep_all && roi), "HIPAC_SCAN_KEEP_ALL cannot be combined with an ROI");
  if (int e = upload_constants(stream)) return e;

  ScanParams p;
  p.rgb = d_rgb, p.H = H, p.W = W, p.pitch = pitch_bytes, p.mask = d_mask, p.mask_pitch = mask_pitch;
  p.P = P, p.S = S, p.nx = nx, p.ny = ny, p.iy_begin = iy_begin;
  OutParams o;
  o.batch_u8 = d_batch_u8, o.batch = (uint16_t*)d_batch, o.layout = layout;
  const int n_cand = nx * ny;

  uint8_t* ws = (uint8_t*)d_workspace;
  uint8_t* flags = ws;
  ws += align_up((size_t)n_cand, 256);
  int32_t* src_idx = (int32_t*)ws;
  ws += align_up((size_t)n_cand * 4, 256);
  int32_t* block_tot = (int32_t*)ws;
  ws += align_up((size_t)((n_cand + kCompactBlock - 1) / kCompactBlock) * 4, 256);

  if (n_cand == 0) {
    HIPAC_CHECK_CUDA(cudaMemsetAsync(d_count, 0, 8, stream));
    return publish_count(d_count, stream);
  }
  if (tissue) {
    tissue_cell_grid(S, P, iy_begin, nx, ny, &tissue->g, &tissue->cy0, &tissue->ncx, &tissue->ncy);
    HIPAC_REQUIRE(tissue->ncy <= 65535, "too many tissue cell rows for one call; split the row range");
  }
  FusedGeom geom;
  const bool fused_ok = n_cand > 0 && fused_geometry(p, &geom) && ((uintptr_t)d_rgb & 15) == 0;
  HIPAC_REQUIRE(mode != HIPAC_SCAN_FUSED || fused_ok,
                "fused scan needs stride % (P/224) == 0, gcd(stride, P) % 32 == 0 and a 16-byte aligned image");
  if (mode != HIPAC_SCAN_DIRECT && fused_ok) {
    return fused_scan_impl(p, o, flags, src_idx, block_tot, d_coords, d_labels, d_count, capacity, ws, stream, keep_all, allow_stream,
                           tissue, roi);
  }
  {
    ProfileScope ps("stats_direct", stream, 0.0);
    k_stats_direct<<<n_cand, 256, 0, stream>>>(p, flags);
  }
  count_launch(1);
  if (tissue)
    if (int e = launch_tissue_filter(p, *tissue, flags, n_cand, stream)) return e;
  if (roi)
    if (int e = launch_roi_filter(p, *roi, flags, n_cand, stream)) return e;
  if (int e = launch_compact(p, flags, n_cand, d_coords, d_labels, src_idx, d_count, capacity, keep_all, block_tot, stream)) return e;
  if (int e = publish_count(d_count, stream)) return e;
  if ((d_batch_u8 || d_batch) && capacity > 0) {
    dim3 grid((unsigned)min(n_cand, capacity), OUT);
    ProfileScope ps("resample_direct", stream, 0.0);
    k_resample_direct<<<grid, 256, 0, stream>>>(p, o, d_coords, d_count, capacity);
    count_launch(1);
  }
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int hipac_tile_scan(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, const uint8_t* d_mask,
                               int64_t mask_pitch, int P, int S, int iy_begin, int iy_end, int32_t* d_coords,
                               uint8_t* d_labels, uint8_t* d_batch_u8, void* d_batch, int layout, int32_t* d_count,
                               int capacity, void* d_workspace, size_t workspace_bytes, int mode, void* stream) {
  return tile_scan_impl(d_rgb, H, W, pitch_bytes, d_mask, mask_pitch, P, S, iy_begin, iy_end, d_coords, d_labels, d_batch_u8, d_batch,
                        layout, d_count, capacity, d_workspace, workspace_bytes, mode, nullptr, nullptr, (cudaStream_t)stream);
}

// hipac_tile_scan_tissue and hipac_tile_scan_roi: the tissue-mask filter (tissue_scale > 0) or the mean > 240 rule
// (tissue_scale = 0, ROI only), then the optional ROI filter
static int tile_scan_filtered(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, const uint8_t* d_mask, int64_t mask_pitch,
                              int P, int S, int iy_begin, int iy_end, int32_t* d_coords, uint8_t* d_labels, uint8_t* d_batch_u8,
                              void* d_batch, int layout, int32_t* d_count, int capacity, void* d_workspace, size_t workspace_bytes,
                              int mode, const uint8_t* d_tissue, int tissue_h, int tissue_w, int64_t tissue_pitch, int tissue_scale,
                              int min_tissue_pixels, const RoiFilter* roi, cudaStream_t stream) {
  if (roi && tissue_scale == 0)
    return tile_scan_impl(d_rgb, H, W, pitch_bytes, d_mask, mask_pitch, P, S, iy_begin, iy_end, d_coords, d_labels, d_batch_u8, d_batch,
                          layout, d_count, capacity, d_workspace, workspace_bytes, mode, nullptr, roi, stream);
  if (int e = tissue_geometry(P, S, tissue_scale)) return e;
  HIPAC_REQUIRE(tissue_h >= 0 && tissue_w >= 0, "negative tissue mask size");
  HIPAC_REQUIRE(d_tissue || (int64_t)tissue_h * tissue_w == 0, "null tissue mask with a nonzero size");
  HIPAC_REQUIRE(tissue_h == 0 || tissue_pitch >= tissue_w, "tissue mask pitch smaller than a row");
  HIPAC_REQUIRE(min_tissue_pixels >= 0, "negative min_tissue_pixels");
  const size_t cells = tissue_cell_bytes(H, W, P, S, iy_begin, iy_end, tissue_scale);
  if (!cells) return -1;
  HIPAC_REQUIRE(d_workspace, "null pointer");
  HIPAC_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "workspace must be 256-byte aligned");
  HIPAC_REQUIRE(workspace_bytes >= hipac_tile_scan_tissue_workspace_bytes(H, W, P, S, iy_begin, iy_end, mode, tissue_scale),
                "workspace too small");
  TissueFilter t{};
  t.mask = d_tissue, t.h = d_tissue ? tissue_h : 0, t.w = d_tissue ? tissue_w : 0, t.pitch = tissue_pitch;
  t.m = tissue_scale, t.min_pixels = min_tissue_pixels;
  t.cells = reinterpret_cast<uint32_t*>(d_workspace);
  return tile_scan_impl(d_rgb, H, W, pitch_bytes, d_mask, mask_pitch, P, S, iy_begin, iy_end, d_coords, d_labels, d_batch_u8, d_batch,
                        layout, d_count, capacity, (uint8_t*)d_workspace + cells, workspace_bytes - cells, mode, &t, roi, stream);
}

extern "C" int hipac_tile_scan_tissue(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, const uint8_t* d_mask,
                                      int64_t mask_pitch, int P, int S, int iy_begin, int iy_end, int32_t* d_coords,
                                      uint8_t* d_labels, uint8_t* d_batch_u8, void* d_batch, int layout, int32_t* d_count,
                                      int capacity, void* d_workspace, size_t workspace_bytes, int mode, const uint8_t* d_tissue,
                                      int tissue_h, int tissue_w, int64_t tissue_pitch, int tissue_scale, int min_tissue_pixels,
                                      void* stream) {
  return tile_scan_filtered(d_rgb, H, W, pitch_bytes, d_mask, mask_pitch, P, S, iy_begin, iy_end, d_coords, d_labels, d_batch_u8,
                            d_batch, layout, d_count, capacity, d_workspace, workspace_bytes, mode, d_tissue, tissue_h, tissue_w,
                            tissue_pitch, tissue_scale, min_tissue_pixels, nullptr, (cudaStream_t)stream);
}

extern "C" size_t hipac_tile_scan_roi_workspace_bytes(int H, int W, int P, int S, int iy_begin, int iy_end, int mode, int tissue_scale) {
  return tissue_scale == 0 ? hipac_tile_scan_workspace_bytes(H, W, P, S, iy_begin, iy_end, mode)
                           : hipac_tile_scan_tissue_workspace_bytes(H, W, P, S, iy_begin, iy_end, mode, tissue_scale);
}

extern "C" int hipac_tile_scan_roi(const uint8_t* d_rgb, int H, int W, int64_t pitch_bytes, const uint8_t* d_mask, int64_t mask_pitch,
                                   int P, int S, int iy_begin, int iy_end, int32_t* d_coords, uint8_t* d_labels, uint8_t* d_batch_u8,
                                   void* d_batch, int layout, int32_t* d_count, int capacity, void* d_workspace, size_t workspace_bytes,
                                   int mode, const uint8_t* d_tissue, int tissue_h, int tissue_w, int64_t tissue_pitch, int tissue_scale,
                                   int min_tissue_pixels, const uint8_t* d_roi, int roi_nx, int roi_ny, int roi_level_shift,
                                   int roi_stride, int roi_patch, int64_t y_origin, void* stream) {
  HIPAC_REQUIRE(!(mode & HIPAC_SCAN_KEEP_ALL), "HIPAC_SCAN_KEEP_ALL cannot be combined with an ROI");
  HIPAC_REQUIRE(d_roi, "null ROI grid");
  HIPAC_REQUIRE(roi_nx > 0 && roi_ny > 0 && (int64_t)roi_nx * roi_ny < ((int64_t)1 << 31), "ROI grid must have 1 to 2^31 - 1 cells");
  HIPAC_REQUIRE(roi_level_shift >= 1 && roi_level_shift <= 16,
                "roi_level_shift = coarse level - fine level must be in [1, 16]: the ROI must come from a coarser level");
  HIPAC_REQUIRE(roi_stride > 0, "roi_stride must be positive");
  HIPAC_REQUIRE(roi_patch > 0, "roi_patch must be positive");
  HIPAC_REQUIRE(y_origin >= 0, "negative y_origin");
  RoiFilter r{};
  r.grid = d_roi, r.nx = roi_nx, r.ny = roi_ny, r.shift = roi_level_shift, r.stride = roi_stride, r.patch = roi_patch;
  r.y_origin = y_origin;
  return tile_scan_filtered(d_rgb, H, W, pitch_bytes, d_mask, mask_pitch, P, S, iy_begin, iy_end, d_coords, d_labels, d_batch_u8,
                            d_batch, layout, d_count, capacity, d_workspace, workspace_bytes, mode, d_tissue, tissue_h, tissue_w,
                            tissue_pitch, tissue_scale, min_tissue_pixels, &r, (cudaStream_t)stream);
}

extern "C" int hipac_upload_rows(void* d_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t row_bytes,
                                 int64_t rows, void* stream) {
  HIPAC_REQUIRE(d_dst && h_src, "null pointer");
  HIPAC_REQUIRE(row_bytes >= 0 && rows >= 0 && dst_pitch >= row_bytes && src_pitch >= row_bytes, "pitch smaller than a row");
  if (row_bytes == 0 || rows == 0) return 0;
  HIPAC_CHECK_CUDA(cudaMemcpy2DAsync(d_dst, (size_t)dst_pitch, h_src, (size_t)src_pitch, (size_t)row_bytes, (size_t)rows,
                                     cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return 0;
}

extern "C" int hipac_tile_scan_set_count_buffer(int32_t* h_count_pinned) {
  g_count_host = h_count_pinned;
  return 0;
}

extern "C" int hipac_tile_scan_wait_count(void) {
  HIPAC_REQUIRE(g_count_host && g_count_event, "no count buffer registered or no scan issued on this thread");
  HIPAC_CHECK_CUDA(cudaEventSynchronize(g_count_event));
  return 0;
}
