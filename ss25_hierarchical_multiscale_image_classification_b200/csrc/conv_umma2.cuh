// The im2col implicit-GEMM kernel on CTA PAIRS (tcgen05 cta_group::2), BN = 256: layer3 and layer4, including their
// stride-2 entry convolutions and the blocks with a fused 1x1 / stride-2 projection (extra K-blocks from a second im2col
// map).  Included by resnet18.cu inside namespace hipac after ConvParams and epilogue_row.
//
// Why pairs here.  With one CTA per tile every 128-pixel tile re-streams the whole weight matrix through its ring: 32 KB of
// weights + 16 KB of activations per 64-wide K-block.  A pair computes TWO pixel tiles against ONE copy of the weights:
// each CTA loads its own activation tile and HALF of the weight rows (16 + 16 KB per K-block), the UMMA is M = 256 x N = 256,
// L2 -> SM traffic drops by a third (measured 16 -> 11 TB/s per launch) and each CTA reads 64 B/clk of operands from shared
// memory instead of 96.  Measured: 5-7 % faster than the single-CTA kernel; what remains is TMA-side (the MMA warp still
// waits on `full` a fifth of the time, the producer on TMA issue).
#pragma once

template <int BN_>
struct Conv2Cfg {
  static constexpr int BN = BN_;
  static constexpr int kBHalfBytes = (BN / 2) * 128;          // this CTA's half of one [BN x 64] weight block
  static constexpr int kStage = kABytes + kBHalfBytes;        // 32 KB
  static constexpr int kStages = 6;                           // 192 KB in flight per SM
  static constexpr int kTmemCols = 2 * BN;                    // the whole TMEM of both SMs
  static constexpr int kSmemBytes = kStages * kStage + 1024 + 256;
  static_assert(BN == 256, "layer3 / layer4 only");
};

template <int BN>
__global__ void __launch_bounds__(conv_threads(BN), 1)
k_conv_umma2(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmA2, const ConvParams p) {
  using Cfg = Conv2Cfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(base + Cfg::kStages * Cfg::kStage);   // leader
  uint64_t* empty = full + Cfg::kStages;                                             // local
  uint64_t* tfull = empty + Cfg::kStages;                                            // local
  uint64_t* tempty = tfull + 2;                                                      // leader
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  ptx::pdl_launch_dependents();
  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    if (p.num_kb2) ptx::prefetch_tensormap(&tmA2);
    for (int s = 0; s < Cfg::kStages; s++) ptx::mbar_init(&full[s], 1), ptx::mbar_init(&empty[s], 1);
    for (int a = 0; a < 2; a++) ptx::mbar_init(&tfull[a], 1), ptx::mbar_init(&tempty[a], 8);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc2(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish2();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  ptx::pdl_wait();
  const int M_total = effective_patches(p.n_dev, p.n_base, p.M_total / p.hw_out) * p.hw_out;
  const int num_m_tiles = (M_total + kBM - 1) / kBM;
  const int num_ptiles = ((num_m_tiles + 1) >> 1) * p.num_n_tiles;       // pair tiles: two pixel tiles x one weight tile
  const int pair0 = blockIdx.x >> 1, pair_step = gridDim.x >> 1;
  // pixel tile of this CTA inside pair tile tp (a phantom second tile of an odd count re-reads the last real one, stores nothing)
  auto tile_of = [&](int tp, int& n_tile, bool& active) {
    const int vt = p.reverse ? num_ptiles - 1 - tp : tp;
    const int m_pair = vt / p.num_n_tiles;
    n_tile = vt - m_pair * p.num_n_tiles;
    int m_tile = 2 * m_pair + (int)rank;
    active = m_tile < num_m_tiles;
    return active ? m_tile : num_m_tiles - 1;
  };

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int tp = pair0; tp < num_ptiles; tp += pair_step) {
      int n_tile;
      bool active;
      const int m0 = tile_of(tp, n_tile, active) * kBM;
      const int img = m0 / p.hw_out, rem = m0 - img * p.hw_out;
      const int p0 = rem / p.wout, q0 = rem - p0 * p.wout;
      const int cw = q0 * p.stride - p.pad_w, ch = p0 * p.stride - p.pad_h;
      for (int kb = 0; kb < p.num_kb + p.num_kb2; kb++) {
        ptx::mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* a_dst = base + stage * Cfg::kStage;
        uint8_t* b_dst = a_dst + kABytes;
        const int tap = kb / p.kc_blocks, kc = kb - tap * p.kc_blocks;
        const int r = tap / p.kw, s = tap - r * p.kw;
        if (ptx::elect_one()) {
          // the leader alone arms the barrier, for both CTAs' bytes (the peer's may land first: the tx-count goes negative and the
          // phase stays open until the leader's arrive).  A remote release-arrive per K-block from the peer costs a MEMBAR.GPU each.
          if (leader) ptx::mbar_arrive_expect_tx(&full[stage], 2 * Cfg::kStage);
          if (kb < p.num_kb)
            ptx::tma2_load_im2col_4d(a_dst, &tmA, &full[stage], kc * 64, cw, ch, img, (uint16_t)s, (uint16_t)r);
          else
            ptx::tma2_load_im2col_4d(a_dst, &tmA2, &full[stage], (kb - p.num_kb) * 64, q0 * p.stride2, p0 * p.stride2, img, 0, 0);
          ptx::tma2_load_2d(b_dst, &tmB, &full[stage], kb * 64, n_tile * BN + (int)rank * (BN / 2));
        }
        __syncwarp();
        if (++stage == Cfg::kStages) stage = 0, phase ^= 1;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader only) =====================
    if (leader) {
      constexpr uint32_t idesc = ptx::make_idesc_bf16(256, BN);
      int stage = 0;
      uint32_t phase = 0, acc = 0, acc_phase = 0;
      for (int tp = pair0; tp < num_ptiles; tp += pair_step) {
        ptx::mbar_wait(&tempty[acc], acc_phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < p.num_kb + p.num_kb2; kb++) {
          ptx::mbar_wait(&full[stage], phase);
          ptx::tc_fence_after();
          const uint32_t a_addr = ptx::smem_u32(base + stage * Cfg::kStage);
          const uint64_t adesc = ptx::make_smem_desc(a_addr, 128), bdesc = ptx::make_smem_desc(a_addr + kABytes, 128);
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; k++) ptx::umma2_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            ptx::umma2_commit_mc(&empty[stage]);
          }
          __syncwarp();
          if (++stage == Cfg::kStages) stage = 0, phase ^= 1;
        }
        if (ptx::elect_one()) ptx::umma2_commit_mc(&tfull[acc]);
        __syncwarp();
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // ===================== epilogue (both CTAs, own 128 accumulator rows) =====================
    const int wq = warp & 3;
    const int row = wq * 32 + lane;
    int it = 0;
    for (int tp = pair0; tp < num_ptiles; tp += pair_step, ++it) {
      const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
      int n_tile;
      bool active;
      const int m = tile_of(tp, n_tile, active) * kBM + row;
      const bool valid = active && m < M_total;
      const size_t off = (size_t)m * p.cout + (size_t)n_tile * BN;
      epilogue_row<BN>(tmem_base + ((uint32_t)(wq * 32) << 16) + acc * BN, p.bias + n_tile * BN,
                       (p.residual && valid) ? p.residual + off : nullptr, p.out + off, p.relu, valid, &tfull[acc], acc_phase);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) ptx::mbar_arrive(&tempty[acc]);
        else ptx::mbar_arrive_cluster(&tempty[acc], 0);
      }
    }
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) ptx::tmem_dealloc2(tmem_base, Cfg::kTmemCols);
}
