// Fused stem: conv1 (7x7 / stride 2 / pad 3, 3 -> 64, folded BN, ReLU) + MaxPool 3x3 / stride 2 / pad 1,
// bf16 space-to-depth batch [n][112][115][16] -> bf16 NHWC [n][56][56][64].  Included by resnet18.cu.
//
// conv1 over the 2x2 space-to-depth image is a 4x4 / stride-1 filter over 16-channel pixels (32 B).  One
// M-tile is ONE conv output row (112 positions of the 128 UMMA rows).  A CTA works on blocks of 8 pooled
// rows = 17 conv rows: a single TMA box brings the 20 space-to-depth rows the block touches into shared
// memory (double buffered across blocks; H padding by TMA zero fill, W padding is stored in the batch),
// and each of the 16 filter taps of each conv row is an UMMA whose A descriptor is that region shifted by
// (row + a) * 115 + b pixels (32-byte rows, 32-byte swizzle).  The weights (64 x 256 bf16 = 32 KB) stay
// resident.  The epilogue never writes the 112 x 112 x 64 conv output: it keeps the running vertical max
// of the current pooled row in shared memory, and every second conv row takes the horizontal 3-max and
// stores one pooled row.  Post-ReLU values are >= 0, so the pool's -inf padding is equivalent to skipping
// the out-of-range taps.
//
// Two CTAs of a cluster work on two blocks with ONE UMMA of M = 256 per tap (tcgen05 cta_group::2, the protocol of
// conv_rows2.cuh): this kernel is bound by shared-memory bandwidth -- per conv row the UMMAs read 16 x (4 KB of A +
// 2 KB of weights), the pooling exchange and the TMA writes another ~22 KB, against 128 B/clk -- and in a pair each CTA
// holds and reads only HALF of the weight rows (16 x 1 KB).  Both CTAs then run the same 17 conv rows per block: for the
// top block of an image row "-1" is computed from the zero-filled halo and the epilogue drops it.
#pragma once

constexpr int kStemPB = 8;                        // pooled rows per block (56 = 7 * 8)
constexpr int kStemRows = 2 * kStemPB + 4;        // space-to-depth rows per block region
constexpr int kStemRegionLoad = kStemRows * kS2dW * 32;
constexpr int kStemRegionBytes = (kStemRegionLoad + 128 * 32 + 1023) / 1024 * 1024;  // + slack for the 128-row UMMA window
constexpr int kStemWBytes = 64 * 256 * 2;
constexpr int kStemVBytes = 112 * 128;            // one conv row of bf16 [112][64]
constexpr int kStemWHalf = kStemWBytes / 2;       // one CTA's 32 weight rows
constexpr int kStemSmem = 2 * kStemRegionBytes + kStemWHalf + 2 * kStemVBytes + 1024 + 256;

struct StemParams {
  int num_blocks;  // n_img * (56 / kStemPB)
  const float* bias;
  __nv_bfloat16* out;  // [n][56][56][64]
  const int* n_dev;    // device-count mode, see effective_patches()
  int n_base;
  int reverse;         // block order, see Launch::reverse
};

using ptx::named_bar_sync;

__device__ __forceinline__ uint4 bf16x8_max(uint4 a, uint4 b) {
  uint4 r;
  const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
  __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; i++) pr[i] = __hmax2(pa[i], pb[i]);
  return r;
}

// producer warp, MMA warp, 16 drain warps (4 per TMEM lane quarter: 16 channels each), 4 pool warps
constexpr int kStemDrainWarps = 16;
constexpr int kStemThreads = 64 + 32 * kStemDrainWarps + 128;

__global__ void __launch_bounds__(kStemThreads, 1)
k_conv1_pool(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const StemParams p) {
  constexpr int kWBlock = kStemWHalf / 4;               // one 64-wide K block of this CTA's weight rows
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = base;                                   // 2 block regions
  uint8_t* sW = base + 2 * kStemRegionBytes;            // resident weights, 4 k-blocks of [32 x 64] (128B swizzle)
  uint8_t* sV = sW + kStemWHalf;                        // 2 x completed vertical max [112][64] bf16 (16B chunks XOR-swizzled)
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sV + 2 * kStemVBytes);   // the leader's
  uint64_t* a_empty = a_full + 2;
  uint64_t* w_full = a_empty + 2;                                          // the leader's
  uint64_t* tfull = w_full + 1;
  uint64_t* tempty = tfull + 2;                                            // the leader's
  uint64_t* v_full = tempty + 2;                                           // vertical max of a pooled row is in sV[buf]
  uint64_t* v_empty = v_full + 2;                                          // ... and has been pooled and stored
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(v_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  ptx::pdl_launch_dependents();
  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    for (int s = 0; s < 2; s++) ptx::mbar_init(&a_full[s], 1), ptx::mbar_init(&a_empty[s], 1);
    ptx::mbar_init(w_full, 1);
    for (int a = 0; a < 2; a++) ptx::mbar_init(&tfull[a], 1), ptx::mbar_init(&tempty[a], 2 * kStemDrainWarps);
    for (int b = 0; b < 2; b++) ptx::mbar_init(&v_full[b], kStemDrainWarps), ptx::mbar_init(&v_empty[b], 4);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc2(tmem_slot, 128);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  constexpr int BLOCKS_PER_IMG = 56 / kStemPB;
  if (warp == 0) {   // resident weights: constant data, loaded before the dependency wait
    if (ptx::elect_one()) {
      if (leader) ptx::mbar_arrive_expect_tx(w_full, kStemWBytes);   // both CTAs' halves
      for (int kb = 0; kb < 4; kb++) ptx::tma2_load_2d(sW + kb * kWBlock, &tmB, w_full, kb * 64, (int)rank * 32);
    }
    __syncwarp();
  }
  ptx::pdl_wait();
  const int num_blocks = effective_patches(p.n_dev, p.n_base, p.num_blocks / BLOCKS_PER_IMG) * BLOCKS_PER_IMG;
  // work items: pairs of consecutive blocks; a phantom second block of an odd count re-reads the last real one and stores
  // nothing
  const int num_items = (num_blocks + 1) >> 1;
  const int item0 = (int)(blockIdx.x >> 1), item_step = (int)(gridDim.x >> 1);
  auto block_of = [&](int it, bool& active) {
    int b = 2 * it + (int)rank;
    active = b < num_blocks;
    if (!active) b = num_blocks - 1;
    return p.reverse ? num_blocks - 1 - b : b;
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    int s = 0;
    uint32_t ph = 0;
    for (int it = item0; it < num_items; it += item_step) {
      bool active;
      const int vb = block_of(it, active);
      const int img = vb / BLOCKS_PER_IMG, py0 = (vb - img * BLOCKS_PER_IMG) * kStemPB;
      ptx::mbar_wait(&a_empty[s], ph ^ 1);
      if (ptx::elect_one()) {
        if (leader) ptx::mbar_arrive_expect_tx(&a_full[s], 2 * kStemRegionLoad);
        ptx::tma2_load_4d(sA + s * kStemRegionBytes, &tmA, &a_full[s], 0, 0, 2 * py0 - 3, img);
      }
      __syncwarp();
      if (++s == 2) s = 0, ph ^= 1;
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (the leader's only) =====================
    if (leader) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(256, 64);
      ptx::mbar_wait(w_full, 0);
      const uint64_t wdesc = ptx::make_smem_desc(ptx::smem_u32(sW), 128);
      int s = 0;
      uint32_t ph = 0, acc = 0, acc_phase = 0;
      for (int it = item0; it < num_items; it += item_step) {
        bool active;
        const int py0 = (block_of(it, active) % BLOCKS_PER_IMG) * kStemPB;
        ptx::mbar_wait(&a_full[s], ph);
        ptx::tc_fence_after();
        const uint64_t rdesc = ptx::make_smem_desc(ptx::smem_u32(sA + s * kStemRegionBytes), 32);
        // conv row 2*py0 - 1 + t; row -1 does not exist: computed and dropped
        for (int t = 0; t <= 2 * kStemPB; t++) {
          ptx::mbar_wait(&tempty[acc], acc_phase ^ 1);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * 64;
          if (ptx::elect_one()) {
#pragma unroll
            for (int a = 0; a < 4; a++)
#pragma unroll
              for (int b = 0; b < 4; b++) {
                const uint64_t ad = rdesc + (uint64_t)(((t + a) * kS2dW + b) * 2), bd = wdesc + (uint64_t)(a * (kWBlock / 16) + b * 2);
                ptx::umma2_bf16(d_tmem, ad, bd, idesc, (a | b) != 0 ? 1u : 0u);
              }
            ptx::umma2_commit_mc(&tfull[acc]);
          }
          __syncwarp();
          acc ^= 1;
          if (acc == 0) acc_phase ^= 1;
        }
        if (ptx::elect_one()) ptx::umma2_commit_mc(&a_empty[s]);
        __syncwarp();
        if (++s == 2) s = 0, ph ^= 1;
      }
    }
  } else if (warp < 2 + kStemDrainWarps) {
    // ===================== drain warps: accumulator + bias -> bf16 -> running vertical max =====================
    // warp (2 + 4*sub + wq) owns TMEM lanes 32*wq.. and channels 16*sub..16*sub+15 of every conv row.  ReLU commutes with
    // the max and with the bf16 rounding, so it is applied once per pooled row (by the pool warps), not per conv row.
    const int wq = warp & 3, sub = (warp - 2) >> 2;
    const int x = wq * 32 + lane;          // conv column of this thread's accumulator row
    const bool valid = x < 112;
    uint32_t acc = 0, acc_phase = 0, closings = 0;
    // bias of this thread's 16 channels and the running vertical max of its conv column live in registers: the
    // accumulator row of lane x is conv column x for EVERY tile, so the vertical 3-max never leaves the thread
    float bias[16];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + sub * 16) + i);
      bias[4 * i] = b.x, bias[4 * i + 1] = b.y, bias[4 * i + 2] = b.z, bias[4 * i + 3] = b.w;
    }
    __nv_bfloat162 vm[8];
    for (int it = item0; it < num_items; it += item_step) {
      bool active;
      const int py0 = (block_of(it, active) % BLOCKS_PER_IMG) * kStemPB;
      const int t_first = py0 == 0 ? 1 : 0;           // first existing conv row of the block: starts the running max
      for (int t = 0; t <= 2 * kStemPB; t++) {
        const bool init = t == t_first;
        const bool closes = t > 0 && (t & 1) == 0;    // conv row 2*py + 1: pooled row py = py0 + t/2 - 1 is complete
        ptx::mbar_wait(&tfull[acc], acc_phase);
        ptx::tc_fence_after();
        uint32_t v[16];
        ptx::tmem_ld_32x32b_x16(tmem_base + ((uint32_t)(wq * 32) << 16) + acc * 64 + sub * 16, v);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) {   // accumulator drained into registers
          if (leader) ptx::mbar_arrive(&tempty[acc]);
          else ptx::mbar_arrive_cluster(&tempty[acc], 0);
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        if (t < t_first) continue;                    // row "-1" of a top block
        __nv_bfloat162 cur[8];  // this pixel's 16 channels: + folded-BN bias (packed fp32 adds), bf16
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const float2 s2 = ptx::fadd2(make_float2(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1])), make_float2(bias[2 * i], bias[2 * i + 1]));
          cur[i] = __floats2bfloat162_rn(s2.x, s2.y);
        }
        if (init) {
#pragma unroll
          for (int i = 0; i < 8; i++) vm[i] = cur[i];
        } else {
#pragma unroll
          for (int i = 0; i < 8; i++) vm[i] = __hmax2(vm[i], cur[i]);
        }
        if (closes) {
          // vertical max complete: hand it to the pool warps through shared memory (double buffered) and restart the
          // running max from this (shared) odd conv row
          const uint32_t b = closings & 1;
          ptx::mbar_wait(&v_empty[b], ((closings >> 1) & 1) ^ 1);
          ++closings;
          if (valid) {
            uint4* mine = reinterpret_cast<uint4*>(sV + b * kStemVBytes + x * 128);
#pragma unroll
            for (int j = 0; j < 2; j++)   // XOR swizzle: conflict-free 16-byte accesses at a 128-byte row stride
              mine[(sub * 2 + j) ^ (x & 7)] = *reinterpret_cast<const uint4*>(&vm[4 * j]);
          }
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&v_full[b]);
#pragma unroll
          for (int i = 0; i < 8; i++) vm[i] = cur[i];
        }
      }
    }
  } else {
    // ===================== pool warps: horizontal 3-max + ReLU -> one pooled row to global memory =====================
    const int pt = threadIdx.x - (64 + 32 * kStemDrainWarps);      // 0..127
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    uint32_t closings = 0;
    for (int it = item0; it < num_items; it += item_step) {
      bool active;
      const int vb = block_of(it, active);
      const int img = vb / BLOCKS_PER_IMG, py0 = (vb - img * BLOCKS_PER_IMG) * kStemPB;
      for (int r = 0; r < kStemPB; r++, closings++) {
        const uint32_t b = closings & 1;
        const uint8_t* buf = sV + b * kStemVBytes;
        ptx::mbar_wait(&v_full[b], (closings >> 1) & 1);
        if (active) {
#pragma unroll
          for (int rep = 0; rep < 2; rep++) {
            const int e = pt + rep * 128;    // (pooled column px, 16-channel quarter): 3-max over conv columns 2px-1, 2px, 2px+1
            if (e < 224) {
              const int px = e >> 2, qtr = e & 3;
              uint4 m[2];
#pragma unroll
              for (int j = 0; j < 2; j++) m[j] = reinterpret_cast<const uint4*>(buf + (2 * px) * 128)[(qtr * 2 + j) ^ ((2 * px) & 7)];
              if (px > 0) {
#pragma unroll
                for (int j = 0; j < 2; j++)
                  m[j] = bf16x8_max(m[j], reinterpret_cast<const uint4*>(buf + (2 * px - 1) * 128)[(qtr * 2 + j) ^ ((2 * px - 1) & 7)]);
              }
#pragma unroll
              for (int j = 0; j < 2; j++)
                m[j] = bf16x8_max(m[j], reinterpret_cast<const uint4*>(buf + (2 * px + 1) * 128)[(qtr * 2 + j) ^ ((2 * px + 1) & 7)]);
              uint4* dst = reinterpret_cast<uint4*>(p.out + (((size_t)img * 56 + py0 + r) * 56 + px) * 64 + qtr * 16);
              dst[0] = bf16x8_max(m[0], zero), dst[1] = bf16x8_max(m[1], zero);   // ReLU
            }
          }
        }
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&v_empty[b]);
      }
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) ptx::tmem_dealloc2(tmem_base, 128);
}
