// Coarse-to-fine cascade: a region of interest (ROI) on a coarse level's candidate grid, built from the scores of its
// survivors, restricts the tile scan of a finer level to the candidates whose footprint meets a set cell.
//   k_roi_clear    zeroes the uint8 [ny][nx] grid
//   k_roi_scatter  one thread per survivor slot; the survivor count is read from device memory when the kernel starts
//                  (min(d_count[0], capacity)), so nothing waits on the host.  A survivor with score >= threshold sets its
//                  cell and every cell within Chebyshev distance `dilate`.
//   k_roi_flags    one thread per fine candidate: walks the closed-form range of coarse cells its footprint overlaps with
//                  positive area and clears bit 0 of its flag unless one of them is set.
// The ROI filter runs between the flag kernel (and the tissue filter) and the compaction of the tile scan, so survivors
// outside the ROI never reach the resample / gather or the network.
#include <algorithm>

#include "tile_scan_shared.cuh"
#include "umma.cuh"

namespace hipac {

__device__ __forceinline__ int64_t floor_div(int64_t a, int64_t b) {   // b > 0
  const int64_t q = a / b;
  return q - ((a % b != 0 && a < 0) ? 1 : 0);
}

__global__ void __launch_bounds__(256) k_roi_clear(uint8_t* __restrict__ grid, int64_t n) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < n; e += (int64_t)gridDim.x * 256) grid[e] = 0;
}

__global__ void __launch_bounds__(256) k_roi_scatter(const int32_t* __restrict__ coords, const float* __restrict__ scores,
                                                     const int32_t* __restrict__ count, int capacity, float threshold, int stride,
                                                     int nx, int ny, int dilate, uint8_t* __restrict__ grid) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int n = min(count[0], capacity);
  for (int s = blockIdx.x * 256 + threadIdx.x; s < n; s += gridDim.x * 256) {
    if (!(scores[s] >= threshold)) continue;
    const int x = coords[2 * s], y = coords[2 * s + 1];
    if (x < 0 || y < 0) continue;
    const int i = x / stride, j = y / stride;
    if (i >= nx || j >= ny) continue;
    const int i0 = (int)max((int64_t)i - dilate, (int64_t)0), i1 = (int)min((int64_t)i + dilate, (int64_t)nx - 1);
    const int j0 = (int)max((int64_t)j - dilate, (int64_t)0), j1 = (int)min((int64_t)j + dilate, (int64_t)ny - 1);
    for (int jj = j0; jj <= j1; jj++)
      for (int ii = i0; ii <= i1; ii++) {
        HIPAC_DEV_ASSERT(ii >= 0 && ii < nx && jj >= 0 && jj < ny);
        grid[(int64_t)jj * nx + ii] = 1;
      }
  }
}

// Cells [c0, c1] whose extent [c*A, c*A + B) overlaps [v, v + p) with positive area: c*A < v + p and c*A + B > v.
__device__ __forceinline__ void roi_cell_range(int64_t v, int p, int64_t A, int64_t B, int n, int* c0, int* c1) {
  *c0 = (int)min(max(floor_div(v - B, A) + 1, (int64_t)0), (int64_t)n);
  *c1 = (int)min(floor_div(v + p - 1, A), (int64_t)n - 1);
}

__global__ void __launch_bounds__(256) k_roi_flags(ScanParams p, RoiFilter r, uint8_t* __restrict__ flags, int n_cand) {
  ptx::pdl_launch_dependents();
  ptx::pdl_wait();
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_cand) return;
  const uint8_t f = flags[idx];
  if (!(f & 1)) return;
  const int ix = idx / p.ny, iyl = idx - ix * p.ny;
  const int64_t x = (int64_t)ix * p.S, y = r.y_origin + (int64_t)(p.iy_begin + iyl) * p.S;
  const int64_t A = (int64_t)r.stride << r.shift, B = (int64_t)r.patch << r.shift;
  int i0, i1, j0, j1;
  roi_cell_range(x, p.P, A, B, r.nx, &i0, &i1);
  roi_cell_range(y, p.P, A, B, r.ny, &j0, &j1);
  for (int j = j0; j <= j1; j++)
    for (int i = i0; i <= i1; i++) {
      HIPAC_DEV_ASSERT(i >= 0 && i < r.nx && j >= 0 && j < r.ny);
      if (r.grid[(int64_t)j * r.nx + i]) return;
    }
  flags[idx] = f & ~1;
}

int launch_roi_filter(const ScanParams& p, const RoiFilter& r, uint8_t* flags, int n_cand, cudaStream_t stream) {
  ProfileScope ps("roi_flags", stream, 0.0);
  HIPAC_CHECK_CUDA(launch_ex(k_roi_flags, dim3((n_cand + 255) / 256), dim3(256), 0, stream, 1, p, r, flags, n_cand));
  count_launch(1);
  return 0;
}

}  // namespace hipac

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace hipac;

extern "C" size_t hipac_roi_grid_bytes(int nx, int ny) {
  if (nx <= 0 || ny <= 0 || (int64_t)nx * ny >= ((int64_t)1 << 31)) {
    set_error("invalid argument: ROI grid must have 1 to 2^31 - 1 cells");
    return 0;
  }
  return (size_t)nx * ny;
}

extern "C" int hipac_roi_grid(const int32_t* d_coords, const float* d_scores, const int32_t* d_count, int capacity, float threshold,
                              int stride, int nx, int ny, int dilate, uint8_t* d_grid, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  HIPAC_REQUIRE(nx > 0 && ny > 0 && (int64_t)nx * ny < ((int64_t)1 << 31), "ROI grid must have 1 to 2^31 - 1 cells");
  HIPAC_REQUIRE(stride > 0, "stride must be positive");
  HIPAC_REQUIRE(capacity >= 0, "negative capacity");
  HIPAC_REQUIRE(dilate >= 0, "negative dilate");
  HIPAC_REQUIRE(d_grid && d_count && (capacity == 0 || (d_coords && d_scores)), "null pointer");
  const int64_t cells = (int64_t)nx * ny;
  {
    ProfileScope ps("roi_clear", stream, (double)cells);
    HIPAC_CHECK_CUDA(launch_ex(k_roi_clear, dim3((unsigned)std::min<int64_t>((cells + 255) / 256, 1024)), dim3(256), 0, stream, 1, d_grid, cells));
  }
  count_launch(1);
  if (capacity > 0) {
    ProfileScope ps("roi_scatter", stream, 0.0);
    HIPAC_CHECK_CUDA(launch_ex(k_roi_scatter, dim3((unsigned)std::min((capacity + 255) / 256, 1024)), dim3(256), 0, stream, 1, d_coords,
                               d_scores, d_count, capacity, threshold, stride, nx, ny, dilate, d_grid));
    count_launch(1);
  }
  return 0;
}
