// Stage 2 of the HiPAC hot path: ResNet18 forward (reference src/models/resnet.py:22-77, i.e. the
// torchvision resnet18 trunk in eval mode + global average pool [+ Linear(512,k)]) as implicit-GEMM
// tcgen05/TMEM kernels.  Activations are bf16 NHWC; eval-mode BatchNorm is folded into the weights
// (fp32 fold, bf16 round) and a per-channel fp32 bias added in the epilogue together with the
// residual and ReLU.  The A operand (im2col of the activations) is produced by TMA im2col loads,
// the B operand (weights, K-major) by tiled TMA loads; accumulators live in TMEM, double buffered
// so the epilogue of tile i overlaps the MMAs of tile i+1.  See DESIGN.md.
#include <cuda.h>

#include <cmath>
#include <cstring>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "resnet18_layers.h"
#include "umma.cuh"

namespace hipac {

// ==========================================================================================
// what the convolution kernels (conv_*.cuh) share
// ==========================================================================================
struct ConvParams {   // the im2col kernel's (conv_umma2.cuh)
  int M_total;       // images * hout * wout (GEMM M)
  int hw_out, wout;  // hout*wout, wout
  int stride, pad_w, pad_h;
  int kw;            // filter width (taps per filter row)
  int kc_blocks;     // 64-channel blocks per tap (cin / 64)
  int num_kb;        // k-blocks per tile from the main operand
  int num_kb2;       // extra k-blocks from the second operand (fused 1x1 projection shortcut), 0 if none
  int stride2;       // traversal stride of the second operand (pad 0, 1x1)
  int num_m_tiles, num_n_tiles;
  int cout;
  int relu;
  const float* bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
  const int* n_dev;  // device-side patch count (null: the host-side sizes above are exact)
  int n_base;        // first patch of this chunk: the kernel works on clamp(*n_dev - n_base, 0, host n) patches
  int reverse;       // walk the tiles from the last to the first (see Launch::reverse)
};

// Device-count mode: the host sizes grids, tensor maps and buffers for a CAPACITY; the number of patches that actually
// exist is read from device memory when the kernel starts, so a whole step can be enqueued without a host round trip.
__device__ __forceinline__ int effective_patches(const int* n_dev, int n_base, int n_cap) {
  if (!n_dev) return n_cap;
  const int n = __ldg(n_dev) - n_base;
  return n < 0 ? 0 : (n < n_cap ? n : n_cap);
}

constexpr int kBM = 128;
constexpr int kS2dW = HIPAC_S2D16_WIDTH;  // 112 + 3 explicit zero columns (2 left, 1 right)
constexpr int kABytes = kBM * 128;  // 128 rows x 64 bf16
// 64-wide tiles have so little MMA work per tile that one epilogue warpgroup cannot keep up: they get two, which
// take alternate tiles (= alternate TMEM accumulator buffers).  Wider tiles keep one (register budget).
__host__ __device__ constexpr int epi_groups(int bn) { return bn == 64 ? 2 : 1; }
__host__ __device__ constexpr int conv_threads(int bn) { return 64 + 128 * epi_groups(bn); }

// 32 consecutive output channels of one output pixel: + folded-BN bias (+ residual, already in registers)
// (+ ReLU) -> bf16, 64-byte store.
__device__ __forceinline__ void epilogue_math32(const uint32_t (&v)[32], const float* __restrict__ bias, const uint4* res,
                                                __nv_bfloat16* __restrict__ out, int relu) {
  const float4* b4 = reinterpret_cast<const float4*>(bias);
  uint4 o[4];
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const float4 b = __ldg(b4 + i);
    float x0 = __uint_as_float(v[4 * i + 0]) + b.x, x1 = __uint_as_float(v[4 * i + 1]) + b.y;
    float x2 = __uint_as_float(v[4 * i + 2]) + b.z, x3 = __uint_as_float(v[4 * i + 3]) + b.w;
    if (res) {
      const uint32_t* rw = reinterpret_cast<const uint32_t*>(&res[i >> 1]) + (i & 1) * 2;
      const __nv_bfloat162 ra = *reinterpret_cast<const __nv_bfloat162*>(&rw[0]);
      const __nv_bfloat162 rb = *reinterpret_cast<const __nv_bfloat162*>(&rw[1]);
      x0 += __bfloat162float(ra.x), x1 += __bfloat162float(ra.y);
      x2 += __bfloat162float(rb.x), x3 += __bfloat162float(rb.y);
    }
    if (relu) x0 = fmaxf(x0, 0.f), x1 = fmaxf(x1, 0.f), x2 = fmaxf(x2, 0.f), x3 = fmaxf(x3, 0.f);
    __nv_bfloat162 lo = __floats2bfloat162_rn(x0, x1), hi = __floats2bfloat162_rn(x2, x3);
    uint32_t* ow = reinterpret_cast<uint32_t*>(&o[i >> 1]) + (i & 1) * 2;
    ow[0] = *reinterpret_cast<uint32_t*>(&lo);
    ow[1] = *reinterpret_cast<uint32_t*>(&hi);
  }
  uint4* dst = reinterpret_cast<uint4*>(out);
#pragma unroll
  for (int i = 0; i < 4; i++) dst[i] = o[i];
}

// Epilogue of one accumulator row (BN channels of one output pixel).  The residual row is fetched into
// registers BEFORE waiting for the accumulator (its address does not depend on the MMAs), so its global-load
// latency hides behind the tile's main loop; TMEM is drained 64 columns per wait.
template <int BN>
__device__ __forceinline__ void epilogue_row(uint32_t tmem_row, const float* __restrict__ bias,
                                             const __nv_bfloat16* __restrict__ residual_row, __nv_bfloat16* __restrict__ out_row,
                                             int relu, bool valid, uint64_t* tfull_bar, uint32_t phase) {
  constexpr bool kPrefetch = BN <= 128;  // 16 B per 8 channels: 32 (BN=64) / 64 (BN=128) registers
  uint4 res[kPrefetch ? BN / 8 : 8];
  const bool has_res = residual_row != nullptr && valid;
  if (kPrefetch && has_res) {
#pragma unroll
    for (int i = 0; i < BN / 8; i++) res[i] = __ldg(reinterpret_cast<const uint4*>(residual_row) + i);
  }
  ptx::mbar_wait(tfull_bar, phase);
  ptx::tc_fence_after();
#pragma unroll
  for (int c0 = 0; c0 < BN; c0 += 64) {
    uint32_t v0[32], v1[32];
    ptx::tmem_ld_32x32b_x32(tmem_row + c0, v0);
    ptx::tmem_ld_32x32b_x32(tmem_row + c0 + 32, v1);
    if (!kPrefetch && has_res) {
#pragma unroll
      for (int i = 0; i < 8; i++) res[i] = __ldg(reinterpret_cast<const uint4*>(residual_row + c0) + i);
    }
    ptx::tmem_ld_wait();
    if (valid) {
      const uint4* r0 = has_res ? &res[kPrefetch ? c0 / 8 : 0] : nullptr;
      epilogue_math32(v0, bias + c0, r0, out_row + c0, relu);
      epilogue_math32(v1, bias + c0 + 32, has_res ? r0 + 4 : nullptr, out_row + c0 + 32, relu);
    }
  }
}

#include "conv_umma2.cuh"
#include "conv_rows2.cuh"
#include "conv_rows2_s2.cuh"
#include "conv_stem.cuh"

// ==========================================================================================
// small memory-bound kernels
// ==========================================================================================
// Global average pool over 7x7 (fp32 accumulate) + optional Linear(512,k) in fp32. One CTA per patch.
__global__ void __launch_bounds__(256) k_avgpool_fc(const __nv_bfloat16* __restrict__ in, float* __restrict__ feats,
                                                    float* __restrict__ logits, const float* __restrict__ fc_w,
                                                    const float* __restrict__ fc_b, int num_classes,
                                                    const int* __restrict__ n_dev, int n_base) {
  const int img = blockIdx.x;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  if (n_dev && img >= __ldg(n_dev) - n_base) return;
  __shared__ float f[512];
  const __nv_bfloat16* src = in + (int64_t)img * 49 * 512;
  for (int c2 = threadIdx.x; c2 < 256; c2 += 256) {
    float s0 = 0.f, s1 = 0.f;
    for (int px = 0; px < 49; px++) {
      const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(src + px * 512 + 2 * c2);
      s0 += __bfloat162float(v.x), s1 += __bfloat162float(v.y);
    }
    s0 *= (1.0f / 49.0f), s1 *= (1.0f / 49.0f);
    f[2 * c2] = s0, f[2 * c2 + 1] = s1;
    feats[(int64_t)img * 512 + 2 * c2] = s0;
    feats[(int64_t)img * 512 + 2 * c2 + 1] = s1;
  }
  if (!logits) return;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int k = warp; k < num_classes; k += 8) {
    float s = 0.f;
    for (int c = lane; c < 512; c += 32) s += f[c] * __ldg(fc_w + k * 512 + c);
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) logits[(int64_t)img * num_classes + k] = s + __ldg(fc_b + k);
  }
}

// k_avgpool_fc of one view of the D4 test-time augmentation (forward_impl with 8 views).  The pooled features of the view
// are computed as in k_avgpool_fc; view 0 stores them into feats, views 1..7 add them to feats (an fp32 running sum in
// view order), and after view 7 the sum is multiplied by 1/8 and k_avgpool_fc's head is applied to it.  The _rn
// intrinsics keep s * (1/49) + acc from being contracted into one FMA, which would round once where the definition
// rounds twice.
__global__ void __launch_bounds__(256) k_avgpool_fc_d4(const __nv_bfloat16* __restrict__ in, float* __restrict__ feats,
                                                       float* __restrict__ logits, const float* __restrict__ fc_w,
                                                       const float* __restrict__ fc_b, int num_classes,
                                                       const int* __restrict__ n_dev, int n_base, int view) {
  const int img = blockIdx.x;
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();   // also orders the read of feats after the previous view's pool
  if (n_dev && img >= __ldg(n_dev) - n_base) return;
  __shared__ float f[512];
  const __nv_bfloat16* src = in + (int64_t)img * 49 * 512;
  float* dst = feats + (int64_t)img * 512;
  for (int c2 = threadIdx.x; c2 < 256; c2 += 256) {
    float s0 = 0.f, s1 = 0.f;
    for (int px = 0; px < 49; px++) {
      const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(src + px * 512 + 2 * c2);
      s0 += __bfloat162float(v.x), s1 += __bfloat162float(v.y);
    }
    s0 = __fmul_rn(s0, 1.0f / 49.0f), s1 = __fmul_rn(s1, 1.0f / 49.0f);
    if (view > 0) s0 = __fadd_rn(dst[2 * c2], s0), s1 = __fadd_rn(dst[2 * c2 + 1], s1);
    if (view == 7) s0 = __fmul_rn(s0, 0.125f), s1 = __fmul_rn(s1, 0.125f);
    f[2 * c2] = s0, f[2 * c2 + 1] = s1;
    dst[2 * c2] = s0;
    dst[2 * c2 + 1] = s1;
  }
  if (view != 7 || !logits) return;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int k = warp; k < num_classes; k += 8) {
    float s = 0.f;
    for (int c = lane; c < 512; c += 32) s += f[c] * __ldg(fc_w + k * 512 + c);
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) logits[(int64_t)img * num_classes + k] = s + __ldg(fc_b + k);
  }
}

// Pixel (i, j) of D4 view v = 4 f + k of a 224 x 224 image x is pixel (a, b) of x, where the view is
// torch.rot90(flip(x, W) if f else x, k, dims=(H, W)).
__device__ __forceinline__ void d4_source(int view, int i, int j, int& a, int& b) {
  const int k = view & 3;
  a = k == 0 ? i : k == 1 ? j : k == 2 ? 223 - i : 223 - j;
  b = k == 0 ? j : k == 1 ? 223 - i : k == 2 ? 223 - j : i;
  if (view & 4) b = 223 - b;
}

// D4 view `view` of a bf16 batch in `layout` (NHWC3 [n,224,224,3] or S2D16 [n,112,115,16]) -> S2D16 [n,112,115,16], the
// stem's operand.  224 is even, so every view maps 2x2 blocks onto 2x2 blocks: output pixel (Y, X) is one input block with
// its four sub-pixels permuted, i.e. one 32-byte S2D16 load (or two 12-byte NHWC3 row runs) and one 32-byte store.  The
// padding columns and channels 12..15 are written as zero whatever the input holds there.  View 0 of NHWC3 is the plain
// repack of the forward.  Device-count mode: only patches < clamp(*n_dev - n_base, 0, n_img) are written.
__global__ void __launch_bounds__(256) k_d4_view(const uint16_t* __restrict__ in, int layout, uint16_t* __restrict__ out, int n_img,
                                                 int view, const int* __restrict__ n_dev, int n_base) {
  const int64_t total = (int64_t)effective_patches(n_dev, n_base, n_img) * 112 * kS2dW;
  // sub-pixel q = dy * 2 + dx of an output block comes from sub-pixel perm[q] of its input block (independent of the block)
  int perm[4];
#pragma unroll
  for (int q = 0; q < 4; q++) {
    int a, b;
    d4_source(view, q >> 1, q & 1, a, b);
    perm[q] = (a & 1) * 2 + (b & 1);
  }
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int X = (int)(t % kS2dW) - 2;
    const int Y = (int)((t / kS2dW) % 112);
    const int64_t img = t / (112 * kS2dW);
    alignas(16) uint16_t v[16] = {};
    if (X >= 0 && X < 112) {
      int a, b;
      d4_source(view, 2 * Y, 2 * X, a, b);
      const int BY = a >> 1, BX = b >> 1;
      alignas(16) uint16_t s[16];   // the input block, channel (sy * 2 + sx) * 3 + c
      if (layout == HIPAC_LAYOUT_S2D16_BF16) {
        const uint4* p = reinterpret_cast<const uint4*>(in + ((img * 112 + BY) * kS2dW + BX + 2) * 16);
        *reinterpret_cast<uint4*>(&s[0]) = __ldg(p);
        *reinterpret_cast<uint4*>(&s[8]) = __ldg(p + 1);
      } else {
#pragma unroll
        for (int sy = 0; sy < 2; sy++) {
          // pixels 2BX, 2BX + 1 of row 2BY + sy: 12 bytes at a multiple of 12 bytes (4-byte aligned)
          const uint32_t* p = reinterpret_cast<const uint32_t*>(in + ((img * 224 + 2 * BY + sy) * 224 + 2 * BX) * 3);
#pragma unroll
          for (int w = 0; w < 3; w++) {
            const uint32_t u = __ldg(p + w);
            s[sy * 6 + 2 * w] = (uint16_t)(u & 0xFFFFu), s[sy * 6 + 2 * w + 1] = (uint16_t)(u >> 16);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 4; q++)
#pragma unroll
        for (int c = 0; c < 3; c++) {
          const int pq = perm[q];   // selects, not a dynamically indexed (local-memory) array
          v[q * 3 + c] = pq == 0 ? s[c] : pq == 1 ? s[3 + c] : pq == 2 ? s[6 + c] : s[9 + c];
        }
    }
    uint4* dst = reinterpret_cast<uint4*>(out + t * 16);
    dst[0] = *reinterpret_cast<uint4*>(&v[0]);
    dst[1] = *reinterpret_cast<uint4*>(&v[8]);
  }
}

// ==========================================================================================
// host: tensor maps, launches
// ==========================================================================================
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeIm2colFn g_encode_im2col = nullptr;
static EncodeTiledFn g_encode_tiled = nullptr;
// Called at the top of every entry point: resolves the driver entry points once per process.
static int init_driver_api() {
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (!(g_encode_im2col && g_encode_tiled)) {
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    HIPAC_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
    HIPAC_REQUIRE(fn && q == cudaDriverEntryPointSuccess, "driver lacks cuTensorMapEncodeIm2col");
    g_encode_im2col = (EncodeIm2colFn)fn;
    HIPAC_CHECK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    HIPAC_REQUIRE(fn && q == cudaDriverEntryPointSuccess, "driver lacks cuTensorMapEncodeTiled");
    g_encode_tiled = (EncodeTiledFn)fn;
  }
  return 0;
}

// What a stage-2 launch needs besides its operands.  Each C entry point builds one and passes it down; forward_impl
// sets n_base per chunk and reverse per launch, the test hooks take all three from their caller.
struct Launch {
  cudaStream_t stream;
  int sms;            // SM count of the current device
  const int* n_dev;   // device-side patch count (device-count mode, see effective_patches) or null
  int n_base;         // first patch of this chunk
  // Boustrophedon tile order across the layers of one forward pass: a layer whose producer wrote images 0..n-1 walks
  // them n-1..0, so its first ~100 MB of reads are the producer's LAST writes and still sit in the 126 MB L2 (with the
  // same order on both sides they would be the oldest, long evicted).
  int reverse;
};

// Input of conv `cs` on n patches, bf16 NHWC [n][hin][hin][cin], as an im2col map: box = 128 output pixels x 64 channels.
static int make_im2col_map(CUtensorMap* map, const void* ptr, int n, const ConvSpec& cs) {
  const int h = cs.hin, w = cs.hin, c = cs.cin;
  cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2};
  int lower[2] = {-cs.pad, -cs.pad};
  int upper[2] = {cs.pad - (cs.k - 1), cs.pad - (cs.k - 1)};
  cuuint32_t estr[4] = {1, (cuuint32_t)cs.stride, (cuuint32_t)cs.stride, 1};
  CUresult r = g_encode_im2col(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, lower, upper,
                               64u, (cuuint32_t)kBM, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeIm2col failed with CUresult " + std::to_string((int)r));
    return -5;
  }
  // Same driver quirk CUTLASS works around (copy_traits_sm90_im2col.hpp): for tensors smaller than 128 KiB
  // drivers <= 13.1 set a descriptor bit that breaks im2col loads.
  int drv = 0;
  cudaDriverGetVersion(&drv);
  if (drv <= 13010 && (size_t)n * h * w * c * 2 < 131072) reinterpret_cast<uint64_t*>(map)[1] &= ~(1ull << 21);
  return 0;
}

// Weights [cout][K] bf16, K-major: box = 64 (K) x bn rows, 128-byte swizzle.
static int make_weight_map(CUtensorMap* map, const void* ptr, int cout, int K, int bn) {
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)cout};
  cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)bn};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return -5;
  }
  return 0;
}

// Activation tensor [n][h][w][c] (bf16) as a tiled 4-D map: box = box_c channels x box_w x box_h pixels x 1 image, element
// stride `es` along w and h.  `what` names the map in the error message.
static int make_act_map(CUtensorMap* map, const void* ptr, int n, int h, int w, int c, int box_c, int box_w, int box_h, int es,
                        CUtensorMapSwizzle swizzle, const char* what) {
  cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)es, (cuuint32_t)es, 1};
  CUresult res = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (res != CUDA_SUCCESS) {
    set_error(std::string("cuTensorMapEncodeTiled (") + what + ") failed with CUresult " + std::to_string((int)res));
    return -5;
  }
  return 0;
}

// One launch of a CTA-pair kernel (clusters of 2) over `pairs` work items: at most one pair per two SMs, the persistent
// pairs loop over the items.
template <typename... KArgs, typename... Args>
static int launch_pairs(const Launch& ctx, void (*kernel)(KArgs...), int pairs, int threads, int smem, const char* name, double flops,
                        const Args&... args) {
  if (int e = ensure_dyn_smem(kernel, smem)) return e;
  const int max_pairs = ctx.sms / 2;
  const int grid = 2 * (pairs < max_pairs ? pairs : max_pairs);
  {
    ProfileScope ps(name, ctx.stream, flops);
    HIPAC_CHECK_CUDA(launch_ex(kernel, dim3((unsigned)grid), dim3((unsigned)threads), smem, ctx.stream, 2, args...));
  }
  count_launch(1);
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// CTA-pair row kernel (conv_rows2.cuh).  weights = [BN][9*KC*64 (+ KDS*64)] K-major at w_ptr; ds_in = block input of the
// fused projection shortcut (KDS = 1) or null.
template <int BN, int KC, int W, int R, int KDS, bool TEPI = (BN == 64)>
static int launch_rows2_t(const Launch& ctx, const void* w_ptr, const float* bias, const void* in, const void* ds_in,
                          const void* residual, void* out, int n, bool relu, const char* name, double flops) {
  using Cfg = Row2Cfg<BN, KC, W, R, KDS, TEPI>;
  const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B;
  CUtensorMap tmA, tmB;
  // the box is one row-tile region: 64 channels x (W + 2) x (R + 2)
  if (int e = make_act_map(&tmA, in, n, W, W, KC * 64, 64, W + 2, R + 2, 1, sw, "region map")) return e;
  if (int e = make_weight_map(&tmB, w_ptr, BN, (9 * KC + KDS) * 64, BN / 2)) return e;
  CUtensorMap tmA2 = tmA, tmO = tmA, tmR = tmA;
  // the 1x1 / stride-2 projection: the box spans 2 (W + 2) x 2 R input pixels with element strides 2, i.e. delivers
  // (W + 2) x R pixels x 64 channels (out-of-range pixels zero filled)
  if (KDS)
    if (int e = make_act_map(&tmA2, ds_in, n, 2 * W, 2 * W, 64, 64, 2 * (W + 2), 2 * R, 2, sw, "strided projection map")) return e;
  if (Cfg::kTmaEpi) {
    // the box is one OUTPUT row tile, 64 channels x W x R (TMA store of the epilogue's staging tile / TMA load of the
    // residual tile)
    if (int e = make_act_map(&tmO, out, n, W, W, BN, 64, W, R, 1, sw, "tile map")) return e;
    tmR = tmO;
    if (residual)
      if (int e = make_act_map(&tmR, residual, n, W, W, BN, 64, W, R, 1, sw, "tile map")) return e;
  }
  RowConvParams p;
  p.n_img = n, p.num_tiles = n * (W / R), p.relu = relu ? 1 : 0;
  p.n_dev = ctx.n_dev, p.n_base = ctx.n_base, p.reverse = ctx.reverse;
  p.bias = bias;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  return launch_pairs(ctx, k_conv3x3_rows2<BN, KC, W, R, KDS, TEPI>, (p.num_tiles + 1) / 2, conv_threads(BN), Cfg::kSmemBytes, name,
                      flops, tmA, tmB, tmA2, tmO, tmR, p);
}

// layer2.0.conv1 (3x3 / stride 2, 64 -> 128, 56x56 -> 28x28) as a parity-split row kernel on CTA pairs (conv_rows2_s2.cuh).
static int launch_rows2_s2(const Launch& ctx, const void* w_ptr, const float* bias, const void* in, void* out, int n, bool relu,
                           const char* name, double flops) {
  using Cfg = S2Cfg;
  const CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B;
  CUtensorMap tmE, tmO, tmB;
  // element strides 2: the boxes deliver Wp x R (even input rows) and Wp x (R + 1) (odd input rows) pixels x 64 channels
  if (int e = make_act_map(&tmE, in, n, 56, 56, 64, 64, 2 * Cfg::Wp, 2 * Cfg::R, 2, sw, "strided projection map")) return e;
  if (int e = make_act_map(&tmO, in, n, 56, 56, 64, 64, 2 * Cfg::Wp, 2 * (Cfg::R + 1), 2, sw, "strided projection map")) return e;
  if (int e = make_weight_map(&tmB, w_ptr, Cfg::BN, 9 * 64, Cfg::BN / 2)) return e;
  RowConvParams p;
  p.n_img = n, p.num_tiles = n * (Cfg::W / Cfg::R), p.relu = relu ? 1 : 0;
  p.bias = bias, p.residual = nullptr, p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.n_dev = ctx.n_dev, p.n_base = ctx.n_base, p.reverse = ctx.reverse;
  return launch_pairs(ctx, k_conv3x3s2_rows2, (p.num_tiles + 1) / 2, conv_threads(128), Cfg::kSmemBytes, name, flops, tmE, tmO, tmB, p);
}

// Fused conv1 + BN + ReLU + maxpool on the S2D16 batch -> [n][56][56][64], on CTA pairs (conv_stem.cuh).
static int run_stem(const Launch& ctx, const uint8_t* d_packed, const PackedLayout& L, const void* in, void* out, int n) {
  CUtensorMap tmA, tmB;
  // S2D16 [n][112][kS2dW][16]: the box is one block region, all kS2dW pixels of kStemRows rows
  if (int e = make_act_map(&tmA, in, n, 112, kS2dW, 16, 16, kS2dW, kStemRows, 1, CU_TENSOR_MAP_SWIZZLE_32B, "stem region map"))
    return e;
  if (int e = make_weight_map(&tmB, d_packed + L.w_off[0], 64, 256, 32)) return e;
  StemParams p;
  p.num_blocks = n * (56 / kStemPB);
  p.n_dev = ctx.n_dev, p.n_base = ctx.n_base, p.reverse = ctx.reverse;
  p.bias = reinterpret_cast<const float*>(d_packed + L.b_off[0]);
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  return launch_pairs(ctx, k_conv1_pool, (p.num_blocks + 1) / 2, kStemThreads, kStemSmem, "conv1_pool_fused",
                      2.0 * n * 112 * 112 * 64 * 147, tmA, tmB, p);
}

// layer3 / layer4 conv `layer` as the im2col GEMM on CTA pairs (conv_umma2.cuh).  With ds_in, the 1x1 / stride-2
// projection shortcut `ds_layer` of the block input ds_in adds its K-blocks (read through a second im2col map) to the same
// accumulator.  Weights [cout][K] at w_ptr, K = the conv's K followed by the shortcut's.
static int launch_conv2(const Launch& ctx, int layer, int ds_layer, const void* w_ptr, const float* bias, const void* in,
                        const void* ds_in, const void* residual, void* out, int n, bool relu, const char* name) {
  const ConvSpec& cs = kConvs[layer];
  const int K = conv_gemm_k(layer) + (ds_in ? conv_gemm_k(ds_layer) : 0);
  ConvParams p;
  p.M_total = n * cs.hout * cs.hout;
  p.hw_out = cs.hout * cs.hout, p.wout = cs.hout;
  p.cout = cs.cout;
  p.relu = relu ? 1 : 0;
  p.bias = bias;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.num_m_tiles = (p.M_total + kBM - 1) / kBM;
  p.n_dev = ctx.n_dev, p.n_base = ctx.n_base, p.reverse = ctx.reverse;
  p.num_kb2 = 0, p.stride2 = 1;
  p.num_n_tiles = cs.cout / 256;
  p.stride = cs.stride, p.pad_w = p.pad_h = cs.pad, p.kw = cs.k, p.kc_blocks = cs.cin / 64, p.num_kb = cs.k * cs.k * p.kc_blocks;
  CUtensorMap tmA, tmB;
  if (int e = make_weight_map(&tmB, w_ptr, cs.cout, K, 128)) return e;   // box of 128 weight rows: each CTA's half
  if (int e = make_im2col_map(&tmA, in, n, cs)) return e;
  CUtensorMap tmA2 = tmA;
  if (ds_in) {
    const ConvSpec& ds = kConvs[ds_layer];
    p.num_kb2 = ds.cin / 64, p.stride2 = ds.stride;
    if (int e = make_im2col_map(&tmA2, ds_in, n, ds)) return e;
  }
  return launch_pairs(ctx, k_conv_umma2<256>, ((p.num_m_tiles + 1) / 2) * p.num_n_tiles, conv_threads(256), Conv2Cfg<256>::kSmemBytes,
                      name, 2.0 * p.M_total * cs.cout * K, tmA, tmB, tmA2, p);
}

// One conv layer of the network on `n` patches, bf16 NHWC in / out.  Not for layer 0 (conv1, which exists only fused with
// the max pool: run_stem) or layer 7 (layer2.0's projection shortcut, which exists only fused: run_conv_ds_fused).
static int run_conv(const Launch& ctx, const uint8_t* d_packed, const PackedLayout& L, int layer, const void* in, const void* residual,
                    void* out, int n, bool relu) {
  const ConvSpec& cs = kConvs[layer];
  const uint8_t* w = d_packed + L.w_off[layer];
  const float* bias = reinterpret_cast<const float*>(d_packed + L.b_off[layer]);
  if (cs.cout == 64)   // layer1: 3x3 / s1 at 56x56
    return launch_rows2_t<64, 1, 56, 2, 0>(ctx, w, bias, in, nullptr, residual, out, n, relu, "conv3x3_c64", 2.0 * n * 56 * 56 * 64 * 576);
  if (cs.cout == 128 && cs.stride == 2) {   // layer2.0.conv1: 3x3 / s2, 64 -> 128
    HIPAC_REQUIRE(residual == nullptr, "layer2.0.conv1 takes no residual");
    return launch_rows2_s2(ctx, w, bias, in, out, n, relu, "conv3x3_c128", 2.0 * n * 28 * 28 * 128 * 576);
  }
  if (cs.cout == 128) {   // layer2: 3x3 / s1 at 28x28; the residual variant has the staged epilogue (see conv_rows2.cuh)
    if (residual)
      return launch_rows2_t<128, 2, 28, 4, 0, true>(ctx, w, bias, in, nullptr, residual, out, n, relu, "conv3x3_c128",
                                                    2.0 * n * 28 * 28 * 128 * 1152);
    return launch_rows2_t<128, 2, 28, 4, 0>(ctx, w, bias, in, nullptr, nullptr, out, n, relu, "conv3x3_c128", 2.0 * n * 28 * 28 * 128 * 1152);
  }
  // layer3 / layer4: im2col on CTA pairs
  static const char* kNames[2][2] = {{"conv3x3_c256", "conv1x1_c256"}, {"conv3x3_c512", "conv1x1_c512"}};
  return launch_conv2(ctx, layer, -1, w, bias, in, nullptr, residual, out, n, relu, kNames[cs.cout == 512][cs.k == 1]);
}

// conv2 of a stage's first block with its projection shortcut fused: out = relu(conv3x3(in) + conv1x1_s2(block_in) + bias).
// Both GEMMs accumulate into the same TMEM tile (the shortcut is extra K-blocks), so the shortcut tensor never exists.
static int run_conv_ds_fused(const Launch& ctx, const uint8_t* d_packed, const PackedLayout& L, int s, const void* in,
                             const void* block_in, void* out, int n) {
  const void* w = d_packed + L.wf_off[s];
  const float* bias = reinterpret_cast<const float*>(d_packed + L.bf_off[s]);
  if (s == 0) {
    // layer2.0: 3x3 128 -> 128 at 28x28 + 1x1/s2 64 -> 128 from the 56x56 block input, on CTA pairs with resident weights
    return launch_rows2_t<128, 2, 28, 4, 1>(ctx, w, bias, in, block_in, nullptr, out, n, true, "conv3x3+ds_c128",
                                            2.0 * n * 28 * 28 * 128 * fused_gemm_k(0));
  }
  // layer3.0 / layer4.0: im2col on CTA pairs, the shortcut from a second im2col map
  static const char* kNames[3] = {"conv3x3+ds_c128", "conv3x3+ds_c256", "conv3x3+ds_c512"};
  return launch_conv2(ctx, fused_conv_layer(s), fused_ds_layer(s), w, bias, in, block_in, nullptr, out, n, true, kNames[s]);
}

static uint16_t host_bf16(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);  // inf / nan passthrough
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// per-chunk activation buffers (bf16 NHWC), sizes per patch
constexpr size_t kActBytes = (size_t)56 * 56 * 64 * 2;   // largest post-pool activation
constexpr size_t kS2dBytes = (size_t)112 * kS2dW * 16 * 2;

static int clamp_chunk(int chunk, int n) {
  if (chunk <= 0) chunk = 4096;
  if (chunk > n) chunk = n;
  return chunk < 1 ? 1 : chunk;
}

}  // namespace hipac

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace hipac;

extern "C" size_t hipac_resnet18_packed_bytes(int num_classes) { return packed_layout(num_classes).total; }

extern "C" int hipac_resnet18_pack(const float* const* t, int num_tensors, int num_classes, float bn_eps, void* h_packed,
                                   size_t packed_bytes) {
  HIPAC_REQUIRE(num_tensors == HIPAC_RESNET18_NUM_TENSORS, "expected 102 tensors (20 x [conv, bn.w, bn.b, bn.mean, bn.var] + fc.w + fc.b)");
  HIPAC_REQUIRE(num_classes >= 0 && num_classes <= 1024, "bad num_classes");
  const PackedLayout L = packed_layout(num_classes);
  HIPAC_REQUIRE(h_packed && packed_bytes >= L.total, "packed buffer too small");
  memset(h_packed, 0, L.total);
  uint8_t* dst = reinterpret_cast<uint8_t*>(h_packed);
  for (int l = 0; l < HIPAC_RESNET18_NUM_CONVS; l++) {
    const ConvSpec& cs = kConvs[l];
    const float *w = t[5 * l], *g = t[5 * l + 1], *b = t[5 * l + 2], *mu = t[5 * l + 3], *var = t[5 * l + 4];
    HIPAC_REQUIRE(w && g && b && mu && var, "null tensor");
    uint16_t* wp = reinterpret_cast<uint16_t*>(dst + L.w_off[l]);
    float* bp = reinterpret_cast<float*>(dst + L.b_off[l]);
    const int K = conv_gemm_k(l);
    for (int o = 0; o < cs.cout; o++) {
      const float scale = g[o] / sqrtf(var[o] + bn_eps);  // eval-mode BN folded in fp32
      bp[o] = b[o] - mu[o] * scale;
      for (int c = 0; c < cs.cin; c++)
        for (int r = 0; r < cs.k; r++)
          for (int s = 0; s < cs.k; s++) {
            const float v = w[(((size_t)o * cs.cin + c) * cs.k + r) * cs.k + s] * scale;
            size_t kidx;
            if (l == 0) {
              // kh = 2a+dy-1, kw = 2b+dx-1 (filter padded to 8x8 with a zero first row/column)
              const int a = (r + 1) >> 1, dy = (r + 1) & 1, bb = (s + 1) >> 1, dx = (s + 1) & 1;
              kidx = (size_t)(a * 4 + bb) * 16 + (dy * 2 + dx) * 3 + c;
            } else {
              kidx = (size_t)(r * cs.k + s) * cs.cin + c;
            }
            wp[(size_t)o * K + kidx] = host_bf16(v);
          }
    }
  }
  for (int s = 0; s < 3; s++) {
    const int lc = fused_conv_layer(s), ld = fused_ds_layer(s);
    const int cout = kConvs[lc].cout, k1 = conv_gemm_k(lc), k2 = conv_gemm_k(ld), kf = k1 + k2;
    const uint16_t* w1 = reinterpret_cast<const uint16_t*>(dst + L.w_off[lc]);
    const uint16_t* w2 = reinterpret_cast<const uint16_t*>(dst + L.w_off[ld]);
    const float *b1 = reinterpret_cast<const float*>(dst + L.b_off[lc]), *b2 = reinterpret_cast<const float*>(dst + L.b_off[ld]);
    uint16_t* wf = reinterpret_cast<uint16_t*>(dst + L.wf_off[s]);
    float* bf = reinterpret_cast<float*>(dst + L.bf_off[s]);
    for (int o = 0; o < cout; o++) {
      memcpy(wf + (size_t)o * kf, w1 + (size_t)o * k1, (size_t)k1 * 2);
      memcpy(wf + (size_t)o * kf + k1, w2 + (size_t)o * k2, (size_t)k2 * 2);
      bf[o] = b1[o] + b2[o];
    }
  }
  if (num_classes > 0) {
    const float *fw = t[100], *fb = t[101];
    HIPAC_REQUIRE(fw && fb, "num_classes > 0 needs fc weight and bias");
    memcpy(dst + L.fc_w_off, fw, (size_t)num_classes * 512 * 4);
    memcpy(dst + L.fc_b_off, fb, (size_t)num_classes * 4);
  }
  return 0;
}

extern "C" size_t hipac_resnet18_workspace_bytes(int n_patches, int chunk) {
  if (n_patches <= 0) return 256;
  const size_t c = (size_t)clamp_chunk(chunk, n_patches);
  // three activation buffers; the S2D16 scratch buffer is needed only when the caller hands the plain NHWC3 layout or asks
  // for the D4 views (sized for it unconditionally: 0.4 MB / patch)
  return c * (3 * kActBytes + kS2dBytes) + 6 * 1024;
}

extern "C" int hipac_resnet18_conv_layer(const void* d_packed, int num_classes, int layer, const void* d_in,
                                         const void* d_residual, void* d_out, int n_patches, int relu, void* stream_, int reverse,
                                         const int32_t* d_count, int n_base) {
  HIPAC_REQUIRE(d_packed && d_in && d_out, "null pointer");
  HIPAC_REQUIRE(layer >= 0 && layer < HIPAC_RESNET18_NUM_CONVS, "layer index out of range");
  HIPAC_REQUIRE(layer != 0, "layer 0 (conv1) runs only fused with the max pool: use hipac_resnet18_stem");
  HIPAC_REQUIRE(layer != 7, "layer 7 (layer2.0.downsample) runs only fused into layer2.0.conv2: use hipac_resnet18_conv_ds_fused");
  HIPAC_REQUIRE(n_patches > 0, "n_patches must be positive");
  HIPAC_REQUIRE(n_base >= 0, "n_base must be non-negative");
  int sms = 0;
  if (int e = init_driver_api()) return e;
  if (int e = device_sm_count(&sms)) return e;
  const PackedLayout L = packed_layout(num_classes);
  return run_conv({(cudaStream_t)stream_, sms, d_count, n_base, reverse != 0}, reinterpret_cast<const uint8_t*>(d_packed), L, layer,
                  d_in, d_residual, d_out, n_patches, relu != 0);
}

extern "C" int hipac_resnet18_conv_ds_fused(const void* d_packed, int num_classes, int stage, const void* d_in, const void* d_block_in,
                                            void* d_out, int n_patches, void* stream_, int reverse, const int32_t* d_count, int n_base) {
  HIPAC_REQUIRE(d_packed && d_in && d_block_in && d_out && n_patches > 0, "bad arguments");
  HIPAC_REQUIRE(stage >= 0 && stage < 3, "stage must be 0 (layer2), 1 (layer3) or 2 (layer4)");
  HIPAC_REQUIRE(n_base >= 0, "n_base must be non-negative");
  int sms = 0;
  if (int e = init_driver_api()) return e;
  if (int e = device_sm_count(&sms)) return e;
  const PackedLayout L = packed_layout(num_classes);
  return run_conv_ds_fused({(cudaStream_t)stream_, sms, d_count, n_base, reverse != 0}, reinterpret_cast<const uint8_t*>(d_packed), L,
                           stage, d_in, d_block_in, d_out, n_patches);
}

extern "C" int hipac_resnet18_stem(const void* d_packed, int num_classes, const void* d_in, void* d_out, int n_patches,
                                   void* stream_, int reverse, const int32_t* d_count, int n_base) {
  HIPAC_REQUIRE(d_packed && d_in && d_out && n_patches > 0, "bad arguments");
  HIPAC_REQUIRE(n_base >= 0, "n_base must be non-negative");
  int sms = 0;
  if (int e = init_driver_api()) return e;
  if (int e = device_sm_count(&sms)) return e;
  const PackedLayout L = packed_layout(num_classes);
  return run_stem({(cudaStream_t)stream_, sms, d_count, n_base, reverse != 0}, reinterpret_cast<const uint8_t*>(d_packed), L, d_in,
                  d_out, n_patches);
}

// views = 1: the plain forward.  views = 8: the D4 test-time augmentation, every chunk runs the network on each of its
// eight views in turn (view kernel into the S2D16 scratch buffer, stem, convs, accumulating pool).
static int forward_impl(const void* d_packed, int num_classes, const void* d_batch, int layout, int n_patches,
                        float* d_feats, float* d_logits, void* d_workspace, size_t workspace_bytes, int chunk,
                        void* stream_, const int* d_count, int views) {
  HIPAC_REQUIRE(n_patches >= 0, "negative n_patches");
  if (n_patches == 0) return 0;
  HIPAC_REQUIRE(d_packed && d_batch && d_feats && d_workspace, "null pointer");
  HIPAC_REQUIRE(layout == HIPAC_LAYOUT_S2D16_BF16 || layout == HIPAC_LAYOUT_NHWC3_BF16, "unknown batch layout");
  HIPAC_REQUIRE(!d_logits || num_classes > 0, "logits requested but the packed weights have no classifier head");
  HIPAC_REQUIRE(workspace_bytes >= hipac_resnet18_workspace_bytes(n_patches, chunk), "workspace too small");
  HIPAC_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "workspace must be 256-byte aligned");
  Launch ctx{(cudaStream_t)stream_, 0, d_count, 0, 0};
  if (int e = init_driver_api()) return e;
  if (int e = device_sm_count(&ctx.sms)) return e;
  const PackedLayout L = packed_layout(num_classes);
  const uint8_t* pk = reinterpret_cast<const uint8_t*>(d_packed);
  const int cmax = clamp_chunk(chunk, n_patches);
  uint8_t* ws = reinterpret_cast<uint8_t*>(d_workspace);
  auto carve = [&](size_t bytes) {
    uint8_t* r = ws;
    ws += align_up(bytes, 1024);
    return r;
  };
  uint8_t* A = carve(cmax * kActBytes);
  uint8_t* B = carve(cmax * kActBytes);
  uint8_t* C = carve(cmax * kActBytes);
  uint8_t* s2d = carve(cmax * kS2dBytes);

  const bool s2d_in = layout == HIPAC_LAYOUT_S2D16_BF16;
  const size_t in_bytes = s2d_in ? kS2dBytes : (size_t)224 * 224 * 3 * 2;   // per patch
  for (int i0 = 0; i0 < n_patches; i0 += cmax) {
    const int n = n_patches - i0 < cmax ? n_patches - i0 : cmax;
    ctx.n_base = i0;
    const uint8_t* chunk_in = reinterpret_cast<const uint8_t*>(d_batch) + (size_t)i0 * in_bytes;
    for (int view = 0; view < views; view++) {
      const void* x0 = chunk_in;   // view 0 of an S2D16 batch is the batch itself
      if (!s2d_in || view > 0) {
        // a plain launch: it starts after the previous view's kernels, whose stem may have read the scratch buffer
        {
          ProfileScope ps("d4_view", ctx.stream, (double)n * (in_bytes + kS2dBytes));
          k_d4_view<<<ctx.sms * 8, 256, 0, ctx.stream>>>(reinterpret_cast<const uint16_t*>(chunk_in), layout,
                                                         reinterpret_cast<uint16_t*>(s2d), n, view, ctx.n_dev, ctx.n_base);
        }
        count_launch(1);
        x0 = s2d;
      }
      // the batch was written in ascending patch order, so the first launch of the chain walks it descending, the next
      // ascending, ...
      int pos = 0;   // position of the next launch in the chain
      auto next = [&] {
        Launch c = ctx;
        c.reverse = pos++ % 2 == 0;
        return c;
      };
      auto conv = [&](int layer, const void* in, const void* res, void* out, bool relu) {
        return run_conv(next(), pk, L, layer, in, res, out, n, relu);
      };
      int e = 0;
      if ((e = run_stem(next(), pk, L, x0, A, n))) return e;
      // layer1 (two basic blocks, identity shortcuts)
      if ((e = conv(1, A, nullptr, B, true)) || (e = conv(2, B, A, C, true))) return e;
      if ((e = conv(3, C, nullptr, B, true)) || (e = conv(4, B, C, A, true))) return e;
      // layer2..4: first block has a strided 1x1 projection shortcut
      for (int s = 0; s < 3; s++) {
        const int l0 = 5 + 5 * s;
        if ((e = conv(l0, A, nullptr, B, true))) return e;           // 3x3 / stride 2
        if ((e = run_conv_ds_fused(next(), pk, L, s, B, A, C, n))) return e;   // 3x3 + 1x1/s2 projection + ReLU, one accumulator
        if ((e = conv(l0 + 3, C, nullptr, B, true)) || (e = conv(l0 + 4, B, C, A, true))) return e;
      }
      const auto* pool_in = reinterpret_cast<const __nv_bfloat16*>(A);
      float* feats = d_feats + (size_t)i0 * 512;
      float* logits = d_logits ? d_logits + (size_t)i0 * num_classes : nullptr;
      const float* fc_w = reinterpret_cast<const float*>(pk + L.fc_w_off);
      const float* fc_b = reinterpret_cast<const float*>(pk + L.fc_b_off);
      if (views == 1) {
        ProfileScope ps_pool("avgpool_fc", ctx.stream, (double)n * (49 * 512 * 2 + 512 * 4));
        HIPAC_CHECK_CUDA(launch_ex(k_avgpool_fc, dim3(n), dim3(256), 0, ctx.stream, 1, pool_in, feats, logits, fc_w, fc_b,
                                   num_classes, ctx.n_dev, ctx.n_base));
      } else {
        ProfileScope ps_pool("avgpool_fc_d4", ctx.stream, (double)n * (49 * 512 * 2 + 2 * 512 * 4));
        HIPAC_CHECK_CUDA(launch_ex(k_avgpool_fc_d4, dim3(n), dim3(256), 0, ctx.stream, 1, pool_in, feats, logits, fc_w, fc_b,
                                   num_classes, ctx.n_dev, ctx.n_base, view));
      }
      count_launch(1);
    }
  }
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int hipac_resnet18_forward(const void* d_packed, int num_classes, const void* d_batch, int layout, int n_patches,
                                      float* d_feats, float* d_logits, void* d_workspace, size_t workspace_bytes, int chunk,
                                      void* stream) {
  return forward_impl(d_packed, num_classes, d_batch, layout, n_patches, d_feats, d_logits, d_workspace, workspace_bytes, chunk,
                      stream, nullptr, 1);
}

extern "C" int hipac_resnet18_forward_dcount(const void* d_packed, int num_classes, const void* d_batch, int layout, int capacity,
                                             const int32_t* d_count, float* d_feats, float* d_logits, void* d_workspace,
                                             size_t workspace_bytes, int chunk, void* stream) {
  HIPAC_REQUIRE(d_count != nullptr, "null device count");
  return forward_impl(d_packed, num_classes, d_batch, layout, capacity, d_feats, d_logits, d_workspace, workspace_bytes, chunk,
                      stream, d_count, 1);
}

extern "C" int hipac_resnet18_forward_d4(const void* d_packed, int num_classes, const void* d_batch, int layout, int n_patches,
                                         const int32_t* d_count, float* d_feats, float* d_logits, void* d_workspace,
                                         size_t workspace_bytes, int chunk, void* stream) {
  return forward_impl(d_packed, num_classes, d_batch, layout, n_patches, d_feats, d_logits, d_workspace, workspace_bytes, chunk,
                      stream, d_count, 8);
}

extern "C" int hipac_batch_d4_view(const void* d_in, int layout, int n_patches, int view, void* d_out, const int32_t* d_count,
                                   int n_base, void* stream) {
  HIPAC_REQUIRE(d_in && d_out, "null pointer");
  HIPAC_REQUIRE(layout == HIPAC_LAYOUT_S2D16_BF16 || layout == HIPAC_LAYOUT_NHWC3_BF16, "unknown batch layout");
  HIPAC_REQUIRE(view >= 0 && view < 8, "view must be in 0..7");
  HIPAC_REQUIRE(n_patches >= 0, "negative n_patches");
  HIPAC_REQUIRE(n_base >= 0, "n_base must be non-negative");
  const uintptr_t in = (uintptr_t)d_in, out = (uintptr_t)d_out;
  const size_t in_bytes = (size_t)n_patches * (layout == HIPAC_LAYOUT_S2D16_BF16 ? kS2dBytes : (size_t)224 * 224 * 3 * 2);
  const size_t out_bytes = (size_t)n_patches * kS2dBytes;
  HIPAC_REQUIRE(n_patches == 0 || in + in_bytes <= out || out + out_bytes <= in, "d_out overlaps d_in");
  if (n_patches == 0) return 0;
  int sms = 0;
  if (int e = device_sm_count(&sms)) return e;
  {
    ProfileScope ps("d4_view", (cudaStream_t)stream, (double)(in_bytes + out_bytes));
    k_d4_view<<<sms * 8, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const uint16_t*>(d_in), layout,
                                                          reinterpret_cast<uint16_t*>(d_out), n_patches, view, d_count, n_base);
  }
  count_launch(1);
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
