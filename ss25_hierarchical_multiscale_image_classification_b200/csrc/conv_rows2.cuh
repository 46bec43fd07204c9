// Row-tile 3x3 / stride-1 / pad-1 convolution on CTA PAIRS (tcgen05 cta_group::2), included by resnet18.cu inside
// namespace hipac after conv_umma2.cuh.
//
// The im2col kernel re-reads every activation byte nine times through L2 (once per filter tap), which
// makes the 64- and 128-channel layers L2-bandwidth bound.  Here one M-tile is R whole image rows in
// PADDED-width coordinates (Wp = W + 2 positions per row, R * Wp <= 128): a single tiled TMA load brings
// the (R + 2) x Wp input pixels of one 64-channel slice into shared memory -- TMA's out-of-bounds zero
// fill materialises the conv padding -- and all nine taps read that ONE staged region through UMMA
// descriptors that differ only in their start address (tap (r, s) starts r * Wp + s pixels = rows of
// 128 B further; tests/test_umma_shift_gpu.py pins that hardware behaviour).  Positions x >= W of each
// padded row produce junk accumulator rows that are simply not stored.
//
// Why pairs.  A cta_group::1 UMMA of M = 128 x N x K = 16 reads (128 + N) * 32 bytes of operands from shared memory in
// N / 2 cycles: 192 B/clk at N = 64 and 128 B/clk at N = 128 against a 128 B/clk shared-memory pipe, so the 64- and
// 128-channel layers are shared-memory bound, and the 128-channel weights (9 * 2 * 16 KB = 288 KB) cannot stay resident,
// so every tile re-streams them from L2.  A CTA pair issues one UMMA of M = 256: each CTA supplies its own 128 rows of A
// (its own tile) but only HALF of the weight rows, i.e. (128 + N/2) * 32 bytes per N / 2 cycles (160 / 96 B/clk), and each
// CTA keeps only half of the weight matrix -- 36 KB (N = 64) or 144..152 KB (N = 128) -- RESIDENT for the lifetime of the
// persistent pair.  The 1x1 / stride-2 projection shortcut of layer2.0 rides along as one more K-block whose A operand is
// a strided tiled TMA box (element strides 2) of the block input.
//
// Pipeline (per CTA, same shared-memory layout in both):
//   warp 0  producer: its own tile's region slices by TMA (cta_group::2 form: the bytes are reported to the LEADER's
//           a_full barrier); waits on its LOCAL a_empty, which the leader's commits reach by multicast
//   warp 1  leader only: waits a_full (armed by the leader's producer alone, for both CTAs' bytes), issues the UMMAs, commits a_empty / tfull to both
//           CTAs; in both CTAs it owns the TMEM allocation (cta_group::2 alloc / dealloc are pair-collective)
//   warps 2.. epilogue: wait the LOCAL tfull, drain their CTA's 128 accumulator rows, arrive on the LEADER's tempty
#pragma once

struct RowConvParams {
  int n_img;
  int num_tiles;  // n_img * (H / R)
  int relu;
  const float* bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
  const int* n_dev;  // device-count mode, see effective_patches()
  int n_base;
  int reverse;       // tile order, see Launch::reverse
};

// bias + residual (16-byte chunk of 8 bf16, already loaded) + ReLU on 8 accumulator columns -> 8 bf16
__device__ __forceinline__ uint4 epilogue_chunk8(const uint32_t* v, const float* __restrict__ bias, uint4 res, bool has_res, int relu) {
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias)), b1 = __ldg(reinterpret_cast<const float4*>(bias) + 1);
  float x[8] = {__uint_as_float(v[0]) + b0.x, __uint_as_float(v[1]) + b0.y, __uint_as_float(v[2]) + b0.z, __uint_as_float(v[3]) + b0.w,
                __uint_as_float(v[4]) + b1.x, __uint_as_float(v[5]) + b1.y, __uint_as_float(v[6]) + b1.z, __uint_as_float(v[7]) + b1.w};
  if (has_res) {
    const __nv_bfloat162* r2 = reinterpret_cast<const __nv_bfloat162*>(&res);
#pragma unroll
    for (int i = 0; i < 4; i++) x[2 * i] += __bfloat162float(r2[i].x), x[2 * i + 1] += __bfloat162float(r2[i].y);
  }
  if (relu) {
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = fmaxf(x[i], 0.f);
  }
  uint4 o;
  __nv_bfloat162 t;
  t = __floats2bfloat162_rn(x[0], x[1]), o.x = *reinterpret_cast<uint32_t*>(&t);
  t = __floats2bfloat162_rn(x[2], x[3]), o.y = *reinterpret_cast<uint32_t*>(&t);
  t = __floats2bfloat162_rn(x[4], x[5]), o.z = *reinterpret_cast<uint32_t*>(&t);
  t = __floats2bfloat162_rn(x[6], x[7]), o.w = *reinterpret_cast<uint32_t*>(&t);
  return o;
}

// TEPI: the epilogue moves through shared-memory staging and TMA (always for BN = 64; for BN = 128 only the RESIDUAL variant,
// whose per-thread 256-byte residual fetch is what the LSU cannot keep up with -- it trades one region stage for a
// single staging tile of two 64-channel halves).  With per-thread stores every epilogue thread owns one output pixel and
// writes its 64 channels (128 bytes) straight to global memory, and fetches the 128 residual bytes the same way: a warp
// instruction touches 32 different 128-byte lines, i.e. 32 LSU wavefronts, 512 wavefronts per warp and tile with a
// residual.  Staged, the residual tile arrives by ONE TMA load into a 128-byte-swizzled buffer, every thread reads /
// rewrites only its own 128-byte row of that buffer (16-byte accesses, conflict free) and the finished tile leaves by ONE
// TMA store.
template <int BN, int KC, int W, int R, int KDS, bool TEPI = (BN == 64)>
struct Row2Cfg {
  static constexpr int Wp = W + 2;
  static constexpr int kRegionRows = 128 + 2 * Wp + 2;
  static constexpr int kRegionBytes = (kRegionRows * 128 + 1023) / 1024 * 1024;
  static constexpr int kLoadBytes = (R + 2) * Wp * 128;     // conv slice: (R + 2) x Wp pixels x 64 channels
  static constexpr int kDsLoadBytes = R * Wp * 128;         // projection slice: R x Wp strided pixels x 64 channels
  static constexpr int kBHalf = BN / 2;                     // weight rows held by one CTA
  static constexpr int kBBlock = kBHalf * 128;              // one (tap, 64-channel slice) block of this CTA's half
  static constexpr int kNumB = 9 * KC + KDS;
  static constexpr int kBBytes = kNumB * kBBlock;
  // 64-channel tiles leave through shared-memory staging + TMA (see TEPI above): [warpgroup][buffer] tiles of R x W x 128 B
  static constexpr bool kTmaEpi = TEPI;
  static constexpr int kTileBytes = R * W * 128;                                  // one 64-channel half of an output tile
  static constexpr int kStageBytes = (kTileBytes + 1023) / 1024 * 1024;
  // BN = 64: [warpgroup][buffer] = 4 tiles; BN = 128: ONE tile of two 64-channel halves
  static constexpr int kStagingBytes = !kTmaEpi ? 0 : (BN == 64 ? 4 : 2) * kStageBytes;
  static constexpr int kFree = 232448 - 1024 - 512 - kBBytes - kStagingBytes;
  static constexpr int kAStages = kFree / kRegionBytes >= 4 ? 4 : kFree / kRegionBytes;
  static constexpr int kTmemCols = 2 * BN;
  static constexpr int kSmemBytes = kAStages * kRegionBytes + kBBytes + kStagingBytes + 1024 + 512;
  static_assert(R * Wp <= 128, "tile does not fit one UMMA M = 128 per CTA");
  static_assert(kAStages >= 2, "need at least two region stages");
  static_assert(kSmemBytes <= 232448, "shared memory budget");
};

template <int BN, int KC, int W, int R, int KDS, bool TEPI = (BN == 64)>
__global__ void __launch_bounds__(conv_threads(BN), 1)
k_conv3x3_rows2(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmO,
                const __grid_constant__ CUtensorMap tmR, const RowConvParams p) {
  using Cfg = Row2Cfg<BN, KC, W, R, KDS, TEPI>;
  constexpr int Wp = Cfg::Wp, H = W, TILES_PER_IMG = H / R, NS = Cfg::kAStages, SLICES = KC + KDS;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = base;
  uint8_t* sB = base + NS * Cfg::kRegionBytes;
  uint8_t* sO = sB + Cfg::kBBytes;                                      // staging tiles (64-channel variant only)
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sO + Cfg::kStagingBytes);   // used in the leader
  uint64_t* a_empty = a_full + 4;                                       // local in each CTA
  uint64_t* b_full = a_empty + 4;                                       // leader
  uint64_t* tfull = b_full + 1;                                         // local
  uint64_t* tempty = tfull + 2;                                         // leader
  uint64_t* st_ready = tempty + 2;                                      // local, [warpgroup][buffer]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(st_ready + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  ptx::pdl_launch_dependents();
  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    if (KDS) ptx::prefetch_tensormap(&tmA2);
    for (int s = 0; s < NS; s++) ptx::mbar_init(&a_full[s], 1), ptx::mbar_init(&a_empty[s], 1);
    ptx::mbar_init(b_full, 1);
    for (int a = 0; a < 2; a++) ptx::mbar_init(&tfull[a], 1), ptx::mbar_init(&tempty[a], 8);
    for (int s = 0; s < 4; s++) ptx::mbar_init(&st_ready[s], 1);
    if (Cfg::kTmaEpi) {
      ptx::prefetch_tensormap(&tmO);
      if (p.residual) ptx::prefetch_tensormap(&tmR);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc2(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();          // barriers of both CTAs initialised before any remote arrive / multicast commit
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0) {   // this CTA's half of the resident weights: constant data, loaded before the dependency wait
    if (ptx::elect_one()) {
      if (leader) ptx::mbar_arrive_expect_tx(b_full, 2 * Cfg::kBBytes);   // the leader alone arms the barrier, for both CTAs' bytes
      for (int kb = 0; kb < Cfg::kNumB; kb++) ptx::tma2_load_2d(sB + kb * Cfg::kBBlock, &tmB, b_full, kb * 64, (int)rank * Cfg::kBHalf);
    }
    __syncwarp();
  }
  ptx::pdl_wait();
  const int num_tiles = effective_patches(p.n_dev, p.n_base, p.n_img) * (p.num_tiles / p.n_img);
  const int num_pairs = (num_tiles + 1) >> 1;
  const int pair0 = blockIdx.x >> 1, pair_step = gridDim.x >> 1;
  // tile of this CTA inside pair-tile tp (a phantom second tile of an odd count re-reads the last real one and stores nothing)
  auto tile_of = [&](int tp, bool& active) {
    int t = 2 * tp + (int)rank;
    active = t < num_tiles;
    if (!active) t = num_tiles - 1;
    return p.reverse ? num_tiles - 1 - t : t;
  };

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    int sa = 0;
    uint32_t pa = 0;
    for (int tp = pair0; tp < num_pairs; tp += pair_step) {
      bool active;
      const int vt = tile_of(tp, active);
      const int img = vt / TILES_PER_IMG, p0 = (vt - img * TILES_PER_IMG) * R;
      for (int sl = 0; sl < SLICES; sl++) {
        ptx::mbar_wait(&a_empty[sa], pa ^ 1);
        if (ptx::elect_one()) {
          const uint32_t bytes = sl < KC ? Cfg::kLoadBytes : Cfg::kDsLoadBytes;
          if (leader) ptx::mbar_arrive_expect_tx(&a_full[sa], 2 * bytes);   // peer bytes may land first: tx-count goes negative, phase stays open
          if (Cfg::kTmaEpi && sl == 0 && active && p.residual != nullptr) {
            // the epilogue's residual tile, pulled into L2 now (NS / SLICES tiles ahead): its staging buffer frees up only one
            // tile ahead, which is less than a loaded DRAM round trip (the epilogue warps were waiting on st_ready)
            ptx::tma_prefetch_4d(&tmR, 0, 0, p0, img);
            if (BN == 128) ptx::tma_prefetch_4d(&tmR, 64, 0, p0, img);
          }
          if (sl < KC) ptx::tma2_load_4d(sA + sa * Cfg::kRegionBytes, &tmA, &a_full[sa], sl * 64, -1, p0 - 1, img);
          else ptx::tma2_load_4d(sA + sa * Cfg::kRegionBytes, &tmA2, &a_full[sa], 0, 0, 2 * p0, img);
        }
        __syncwarp();
        if (++sa == NS) sa = 0, pa ^= 1;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(256, BN);
      int sa = 0;
      uint32_t pa = 0, acc = 0, acc_phase = 0;
      ptx::mbar_wait(b_full, 0);
      ptx::tc_fence_after();
      const uint64_t b_all = ptx::make_smem_desc(ptx::smem_u32(sB), 128);
      for (int tp = pair0; tp < num_pairs; tp += pair_step) {
        ptx::mbar_wait(&tempty[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
        for (int sl = 0; sl < SLICES; sl++) {
          ptx::mbar_wait(&a_full[sa], pa);
          ptx::tc_fence_after();
          const uint64_t a_region = ptx::make_smem_desc(ptx::smem_u32(sA + sa * Cfg::kRegionBytes), 128);
          if (ptx::elect_one()) {
            if (sl < KC) {
#pragma unroll
              for (int tap = 0; tap < 9; tap++) {
                const uint64_t adesc = a_region + (uint64_t)(((tap / 3) * Wp + tap % 3) * 8);
                const uint64_t bdesc = b_all + (uint64_t)((tap * KC + sl) * (Cfg::kBBlock >> 4));
#pragma unroll
                for (int k = 0; k < 4; k++) ptx::umma2_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (sl | tap | k) != 0 ? 1u : 0u);
              }
            } else {
              const uint64_t bdesc = b_all + (uint64_t)(9 * KC * (Cfg::kBBlock >> 4));
#pragma unroll
              for (int k = 0; k < 4; k++) ptx::umma2_bf16(d_tmem, a_region + 2 * k, bdesc + 2 * k, idesc, 1u);
            }
            ptx::umma2_commit_mc(&a_empty[sa]);
          }
          __syncwarp();
          if (++sa == NS) sa = 0, pa ^= 1;
        }
        if (ptx::elect_one()) ptx::umma2_commit_mc(&tfull[acc]);
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if constexpr (Cfg::kTmaEpi && BN == 128) {
    // ===================== epilogue, 128 channels with residual: one staging tile of two 64-channel halves =====================
    // thread 0 owns the bulk groups: store of tile j -> wait until it has been read -> residual load of tile j + 1 into the
    // same buffer (the MMAs of tile j + 1 run meanwhile: the accumulators are double buffered in TMEM)
    const int wq = warp & 3;
    const int gt = threadIdx.x - 64;
    const int pos = wq * 32 + lane;
    const int rr = pos / Wp, x = pos - rr * Wp;
    const bool in_tile = rr < R && x < W;
    const int srow = rr * W + x;
    const bool has_res = p.residual != nullptr;
    uint64_t* ready = st_ready;
    auto prepare = [&](int tp) {
      bool active;
      const int vt = tile_of(tp, active);
      if (has_res && active) {
        const int img = vt / TILES_PER_IMG, p0 = (vt - img * TILES_PER_IMG) * R;
        ptx::mbar_arrive_expect_tx(&ready[0], 2 * Cfg::kTileBytes);
        ptx::tma_load_4d(sO, &tmR, &ready[0], 0, 0, p0, img);
        ptx::tma_load_4d(sO + Cfg::kStageBytes, &tmR, &ready[0], 64, 0, p0, img);
      } else {
        ptx::mbar_arrive(&ready[0]);
      }
    };
    if (gt == 0 && pair0 < num_pairs) prepare(pair0);
    int it = 0;
    for (int tp = pair0; tp < num_pairs; tp += pair_step, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      bool active;
      const int vt = tile_of(tp, active);
      ptx::mbar_wait(&ready[0], it & 1);
      ptx::mbar_wait(&tfull[acc], acc_phase);
      ptx::tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * BN;
#pragma unroll
      for (int half = 0; half < 2; half++) {
        uint32_t v0[32], v1[32];
        ptx::tmem_ld_32x32b_x32(trow + half * 64, v0);
        ptx::tmem_ld_32x32b_x32(trow + half * 64 + 32, v1);
        ptx::tmem_ld_wait();
        if (half == 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (leader) ptx::mbar_arrive(&tempty[acc]);
            else ptx::mbar_arrive_cluster(&tempty[acc], 0);
          }
        }
        if (in_tile && active) {
          uint4* row = reinterpret_cast<uint4*>(sO + half * Cfg::kStageBytes + srow * 128);
#pragma unroll
          for (int i = 0; i < 8; i++) {
            const int ph = i ^ (srow & 7);
            uint4 res = make_uint4(0u, 0u, 0u, 0u);
            if (has_res) res = row[ph];
            row[ph] = epilogue_chunk8(i < 4 ? &v0[8 * i] : &v1[8 * (i - 4)], p.bias + half * 64 + 8 * i, res, has_res, p.relu);
          }
        }
      }
      ptx::fence_proxy_async();
      ptx::named_bar_sync(1, 128);
      if (gt == 0) {
        if (active) {
          const int img = vt / TILES_PER_IMG, p0 = (vt - img * TILES_PER_IMG) * R;
          ptx::tma_store_4d(&tmO, sO, 0, 0, p0, img);
          ptx::tma_store_4d(&tmO, sO + Cfg::kStageBytes, 64, 0, p0, img);
        }
        ptx::bulk_commit_group();
        if (tp + pair_step < num_pairs) {
          ptx::bulk_wait_group_read<0>();
          prepare(tp + pair_step);
        }
      }
    }
    if (gt == 0) ptx::bulk_wait_group<0>();
  } else if constexpr (Cfg::kTmaEpi) {
    // ===================== epilogue, 64 channels: TMEM -> staging tile (residual in place) -> TMA store =====================
    // Two staging buffers per epilogue warpgroup: the store of tile j and the residual load of tile j + 1 overlap the math
    // of tile j.  The accumulator-drained arrive goes to the LEADER's tempty barrier.
    const int wq = warp & 3;
    const int grp = (warp - 2) >> 2;
    const int gt = threadIdx.x - 64 - 128 * grp;
    const int pos = wq * 32 + lane;
    const int rr = pos / Wp, x = pos - rr * Wp;
    const bool in_tile = rr < R && x < W;
    const int srow = rr * W + x;
    const bool has_res = p.residual != nullptr;
    uint8_t* stage0 = sO + grp * 2 * Cfg::kStageBytes;
    uint64_t* ready = st_ready + grp * 2;
    const int first = pair0 + grp * pair_step, step = 2 * pair_step;
    auto prepare = [&](int tp, int b) {
      bool active;
      const int vt = tile_of(tp, active);
      if (has_res && active) {
        const int img = vt / TILES_PER_IMG, p0 = (vt - img * TILES_PER_IMG) * R;
        ptx::mbar_arrive_expect_tx(&ready[b], Cfg::kTileBytes);
        ptx::tma_load_4d(stage0 + b * Cfg::kStageBytes, &tmR, &ready[b], 0, 0, p0, img);
      } else {
        ptx::mbar_arrive(&ready[b]);
      }
    };
    if (gt == 0 && first < num_pairs) prepare(first, 0);
    int j = 0;
    for (int tp = first; tp < num_pairs; tp += step, ++j) {
      const int b = j & 1;
      const uint32_t acc = grp, acc_phase = j & 1;
      bool active;
      const int vt = tile_of(tp, active);
      uint8_t* buf = stage0 + b * Cfg::kStageBytes;
      // the NEXT tile's residual goes into the other buffer now, a whole group iteration ahead: that buffer's store (end of
      // the previous iteration) only has to have been read out of shared memory
      if (gt == 0 && tp + step < num_pairs) {
        ptx::bulk_wait_group_read<0>();
        prepare(tp + step, b ^ 1);
      }
      ptx::mbar_wait(&ready[b], (j >> 1) & 1);
      ptx::mbar_wait(&tfull[acc], acc_phase);
      ptx::tc_fence_after();
      uint32_t v0[32], v1[32];
      const uint32_t trow = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * BN;
      ptx::tmem_ld_32x32b_x32(trow, v0);
      ptx::tmem_ld_32x32b_x32(trow + 32, v1);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) ptx::mbar_arrive(&tempty[acc]);
        else ptx::mbar_arrive_cluster(&tempty[acc], 0);
      }
      if (in_tile && active) {
        uint4* row = reinterpret_cast<uint4*>(buf + srow * 128);
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int ph = i ^ (srow & 7);
          uint4 res = make_uint4(0u, 0u, 0u, 0u);
          if (has_res) res = row[ph];
          row[ph] = epilogue_chunk8(i < 4 ? &v0[8 * i] : &v1[8 * (i - 4)], p.bias + 8 * i, res, has_res, p.relu);
        }
      }
      ptx::fence_proxy_async();
      ptx::named_bar_sync(1 + grp, 128);
      if (gt == 0) {
        if (active) {
          const int img = vt / TILES_PER_IMG, p0 = (vt - img * TILES_PER_IMG) * R;
          ptx::tma_store_4d(&tmO, buf, 0, 0, p0, img);
        }
        ptx::bulk_commit_group();
      }
    }
    if (gt == 0) ptx::bulk_wait_group<0>();
  } else {
    // ===================== epilogue (both CTAs, own 128 accumulator rows) =====================
    const int wq = warp & 3;
    const int pos = wq * 32 + lane;
    const int rr = pos / Wp, x = pos - rr * Wp;
    const bool in_tile = rr < R && x < W;
    const int grp = (warp - 2) >> 2;
    int it = 0;
    for (int tp = pair0; tp < num_pairs; tp += pair_step, ++it) {
      if (epi_groups(BN) == 2 && (it & 1) != grp) continue;
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      bool active;
      const int vt = tile_of(tp, active);
      const int img = vt / TILES_PER_IMG, p0 = (vt - img * TILES_PER_IMG) * R;
      const size_t pix = ((size_t)img * H + p0 + rr) * W + x;
      const bool valid = in_tile && active;
      epilogue_row<BN>(tmem_base + ((uint32_t)(wq * 32) << 16) + acc * BN, p.bias, (p.residual && valid) ? p.residual + pix * BN : nullptr,
                       p.out + pix * BN, p.relu, valid, &tfull[acc], acc_phase);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) ptx::mbar_arrive(&tempty[acc]);
        else ptx::mbar_arrive_cluster(&tempty[acc], 0);
      }
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();          // both CTAs are done with each other's shared memory and TMEM
  if (warp == 1) ptx::tmem_dealloc2(tmem_base, Cfg::kTmemCols);
}
