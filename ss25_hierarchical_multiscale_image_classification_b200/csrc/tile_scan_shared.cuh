// Types shared by the direct and fused stage-1 kernels.
#pragma once
#include "common.cuh"

namespace hipac {

struct CoeffSet {       // Pillow 22-bit fixed-point triangle weights for one integer scale
  int32_t interior[16]; // 2*scale taps
  int32_t left[12];     // output 0   (3*scale/2 taps)
  int32_t right[12];    // output 223 (3*scale/2 taps)
};

struct ScanParams {
  const uint8_t* rgb;   // [H][pitch] RGB bytes
  int H, W;
  int64_t pitch;
  const uint8_t* mask;  // [H][mask_pitch] or null
  int64_t mask_pitch;
  int P, S;             // patch size, stride
  int nx, ny;           // candidate grid of this call: nx columns, ny rows starting at iy_begin
  int iy_begin;
};

struct OutParams {
  uint8_t* batch_u8;    // [cap][224][224][3] or null
  uint16_t* batch;      // bf16 bits, layout below, or null
  int layout;
};

// Tissue-mask filter (tissue.cu): mask pixel (u, v) covers level pixels [u*m, u*m+m) x [v*m, v*m+m) of the call's image.
struct TissueFilter {
  const uint8_t* mask;  // [h][pitch], > 0 = tissue
  int h, w;
  int64_t pitch;
  int m, min_pixels;
  int g, cy0, ncx, ncy; // cells of g = gcd(S, P) level pixels: stored cell rows [cy0, cy0 + ncy), columns [0, ncx)
  uint32_t* cells;      // [ncy][ncx] tissue pixel counts (workspace)
};

// The cell grid a candidate range [iy_begin, iy_begin + ny) x [0, nx) reads: every cell of every candidate footprint.
void tissue_cell_grid(int S, int P, int iy_begin, int nx, int ny, int* g, int* cy0, int* ncx, int* ncy);
// k_tissue_cells + k_tissue_flags: rewrites bit 0 of every flag with the tissue-mask rule (after the flag kernel).
int launch_tissue_filter(const ScanParams& p, const TissueFilter& t, uint8_t* flags, int n_cand, cudaStream_t stream);

// Region of interest from a coarser level (cascade.cu): cell (i, j) of the coarse candidate grid covers the fine-level pixels
// [i*stride << shift, (i*stride + patch) << shift) on each axis.
struct RoiFilter {
  const uint8_t* grid;  // [ny][nx], nonzero = set
  int nx, ny;
  int shift;            // coarse level - fine level, >= 1
  int stride, patch;    // S_c, P_c of the coarse level
  int64_t y_origin;     // fine-level row of the scanned image's row 0
};
// k_roi_flags: clears bit 0 of every candidate whose footprint meets no set cell (after the tissue filter, before compaction).
int launch_roi_filter(const ScanParams& p, const RoiFilter& r, uint8_t* flags, int n_cand, cudaStream_t stream);

}  // namespace hipac
