// Macenko stain normalisation: estimate a slide's H&E stain matrix from a thumbnail, then re-express every patch in a
// reference stain.  The contract is torchstain's NumpyMacenkoNormalizer (Io, alpha, beta), with the matrix estimated once
// per slide; oracle/stain.py restates it in numpy and the tests compare against it.
//
// Estimation (hipac_stain_estimate), all on the caller's stream, no host wait, no floating-point atomics, so every run
// (and every rank of a sharded run) gets the same bits:
//   k_stain_sums    per block, fp64: ODhat count and per-channel OD sums (OD = -log((I + 1) / Io), ODhat = all three >= beta)
//   k_stain_cov     per block: the six centred products of ODhat (every block first forms the mean from the fixed-order
//                   sum of the block partials, as np.cov centres)
//   k_stain_eig     one thread: covariance / (n - 1), cyclic Jacobi, eigenpairs ascending, E = the two largest
//   k_stain_phi     key of phi = atan2(T1, T0) per pixel (T = OD . E), +inf for pixels outside ODhat
//   k_stain_hist / k_stain_pick   radix select, 8 passes of 8 bits over order-preserving 64-bit keys: the ranks floor(h) and
//                   floor(h) + 1 of two percentiles in the same passes, n read from device memory
//   k_stain_he      one thread: numpy's _lerp of the percentiles, vMin / vMax, H first; P = (HE^T HE)^-1 HE^T
//   k_stain_conc    keys of C = P . OD per pixel (all pixels), both rows; then the 99th percentiles by the same select
//   k_stain_finish  one thread: the stain block
// Normaliser (hipac_stain_normalizer), one block: the parameter block (valid, Io, M, od) from a source and a target.
// Apply (hipac_stain_apply), the hot path: per CTA the tables A[c][j][v] = M[c][j] * od[v] in shared memory; per pixel and
// channel y = (A[c][0][r] + A[c][1][g]) + A[c][2][b] and out = #{v in 0..254 : y <= od[v]} (= trunc(min(255, Io exp(-y))),
// found from an fp32 guess confirmed by fp64 comparisons), then optionally ToTensor/Normalize to bf16 NHWC3 or S2D16.
#include <algorithm>
#include <cmath>

#include "common.cuh"

namespace hipac {

void host_normalize_lut_bf16(uint16_t* lut);   // tile_scan.cu: stage 1's ToTensor/Normalize table

#define STAIN_THREADS 256         // threads per CTA of every multi-thread stain kernel
#define STAIN_RED_BLOCKS 512      // CTAs of the two fp64 reductions: fixed, so the summation order never depends on the device
#define STAIN_APPLY_CTAS_PER_SM 4 // persistent grid of the apply kernel

constexpr int kTargets = 4;        // ranks selected at once: floor(h) and floor(h) + 1 of two percentiles
__device__ constexpr double kHeRef[3][2] = {{0.5626, 0.2159}, {0.7201, 0.8012}, {0.4062, 0.5581}};   // torchstain's target
__device__ constexpr double kMaxCRef[2] = {1.9705, 1.0308};

struct StainState {
  double E[3][2];                 // the two principal eigenvectors (second largest, largest)
  double he[3][2];
  double P[2][3];
  double gamma[2];                // lerp weight of each percentile
  unsigned long long prefix[kTargets];   // radix select: key bits fixed so far
  unsigned int rank[kTargets];    // rank still to find among the keys with that prefix
  int arr[kTargets];              // 0: keys_a, 1: keys_b
  long long n_hat;
  int valid;
};

__device__ __forceinline__ unsigned long long key_of(double d) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(d);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double double_of(unsigned long long k) {
  return __longlong_as_double((long long)((k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k));
}
constexpr unsigned long long kInfKey = 0xFFF0000000000000ull;   // key_of(+inf)

// numpy's _lerp: a + (b - a) * t, or b - (b - a) * (1 - t) for t >= 0.5
__device__ __forceinline__ double np_lerp(double a, double b, double t) {
  const double d = __dsub_rn(b, a);
  return t >= 0.5 ? __dsub_rn(b, __dmul_rn(d, __dsub_rn(1.0, t))) : __dadd_rn(a, __dmul_rn(d, t));
}

// Targets 2p, 2p + 1 = ranks floor(h), floor(h) + 1 of percentile q (as a fraction) of n keys of array `arr`
// (numpy's "linear" method: h = (n - 1) q; both ranks n - 1 when h >= n - 1).
__device__ void set_percentile(StainState* st, int p, long long n, double q, int arr) {
  const double h = __dmul_rn((double)(n - 1), q);
  long long lo, hi;
  double gamma;
  if (n <= 0) lo = hi = 0, gamma = 0.0;
  else if (h >= (double)(n - 1)) lo = hi = n - 1, gamma = __dadd_rn(h, 1.0);   // numpy: previous index -1
  else lo = (long long)floor(h), hi = lo + 1, gamma = __dsub_rn(h, (double)lo);
  st->gamma[p] = gamma;
  st->rank[2 * p] = (unsigned)lo, st->rank[2 * p + 1] = (unsigned)hi;
  st->prefix[2 * p] = st->prefix[2 * p + 1] = 0;
  st->arr[2 * p] = st->arr[2 * p + 1] = arr;
}

__device__ __forceinline__ double percentile_of(const StainState* st, int p) {
  return np_lerp(double_of(st->prefix[2 * p]), double_of(st->prefix[2 * p + 1]), st->gamma[p]);
}

// P = (HE^T HE)^-1 HE^T by the documented sequence (rows summed 0, 1, 2, every operation rounded on its own); returns det
__device__ double pinv_fixed(const double he[3][2], double P[2][3]) {
  double g[2][2];
  for (int i = 0; i < 2; i++)
    for (int j = 0; j < 2; j++)
      g[i][j] = __dadd_rn(__dadd_rn(__dmul_rn(he[0][i], he[0][j]), __dmul_rn(he[1][i], he[1][j])), __dmul_rn(he[2][i], he[2][j]));
  const double det = __dsub_rn(__dmul_rn(g[0][0], g[1][1]), __dmul_rn(g[0][1], g[0][1]));
  const double inv[2][2] = {{__ddiv_rn(g[1][1], det), __ddiv_rn(-g[0][1], det)}, {__ddiv_rn(-g[0][1], det), __ddiv_rn(g[0][0], det)}};
  for (int i = 0; i < 2; i++)
    for (int j = 0; j < 3; j++) P[i][j] = __dadd_rn(__dmul_rn(inv[i][0], he[j][0]), __dmul_rn(inv[i][1], he[j][1]));
  return det;
}

struct StainImage {
  const uint8_t* rgb;
  int H, W;
  int64_t pitch;
  int io;
  double beta;
};

__device__ __forceinline__ void fill_od(double* s_od, int io) {
  for (int v = threadIdx.x; v < 256; v += blockDim.x) s_od[v] = -log(__ddiv_rn((double)(v + 1), (double)io));
}

__device__ __forceinline__ void pixel_od(const StainImage& im, long long i, const double* s_od, double od[3]) {
  const int y = (int)(i / im.W), x = (int)(i - (long long)y * im.W);
  HIPAC_DEV_ASSERT(y >= 0 && y < im.H && x >= 0 && x < im.W);
  const uint8_t* px = im.rgb + (int64_t)y * im.pitch + (int64_t)x * 3;
  od[0] = s_od[px[0]], od[1] = s_od[px[1]], od[2] = s_od[px[2]];
}

// fixed-order tree sum of s[k][0..STAIN_THREADS) for k < K, result in s[k][0]
template <int K>
__device__ __forceinline__ void block_sum(double (*s)[STAIN_THREADS]) {
  for (int w = STAIN_THREADS / 2; w > 0; w >>= 1) {
    __syncthreads();
    if (threadIdx.x < w)
      for (int k = 0; k < K; k++) s[k][threadIdx.x] = __dadd_rn(s[k][threadIdx.x], s[k][threadIdx.x + w]);
  }
  __syncthreads();
}

// the pixels of block b: a contiguous range, each thread walks it with stride STAIN_THREADS
__device__ __forceinline__ void block_range(long long n, long long& i0, long long& i1) {
  const long long per = (n + gridDim.x - 1) / gridDim.x;
  i0 = std::min(n, (long long)blockIdx.x * per), i1 = std::min(n, i0 + per);
}

__global__ void __launch_bounds__(STAIN_THREADS) k_stain_sums(const StainImage im, double* __restrict__ part) {
  __shared__ double s_od[256];
  __shared__ double s[4][STAIN_THREADS];
  fill_od(s_od, im.io);
  __syncthreads();
  long long i0, i1;
  block_range((long long)im.H * im.W, i0, i1);
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long i = i0 + threadIdx.x; i < i1; i += STAIN_THREADS) {
    double od[3];
    pixel_od(im, i, s_od, od);
    if (od[0] >= im.beta && od[1] >= im.beta && od[2] >= im.beta) {
      acc[0] = __dadd_rn(acc[0], 1.0);
      for (int c = 0; c < 3; c++) acc[c + 1] = __dadd_rn(acc[c + 1], od[c]);
    }
  }
  for (int k = 0; k < 4; k++) s[k][threadIdx.x] = acc[k];
  block_sum<4>(s);
  if (threadIdx.x < 4) part[blockIdx.x * 4 + threadIdx.x] = s[threadIdx.x][0];
}

// sum over the STAIN_RED_BLOCKS partials in block order
__device__ __forceinline__ double partial_sum(const double* part, int stride, int k) {
  double t = 0.0;
  for (int b = 0; b < STAIN_RED_BLOCKS; b++) t = __dadd_rn(t, part[b * stride + k]);
  return t;
}

__global__ void __launch_bounds__(STAIN_THREADS) k_stain_cov(const StainImage im, const double* __restrict__ part1,
                                                             double* __restrict__ part2) {
  __shared__ double s_od[256];
  __shared__ double s_mean[4];
  __shared__ double s[6][STAIN_THREADS];
  fill_od(s_od, im.io);
  if (threadIdx.x < 4) s_mean[threadIdx.x] = partial_sum(part1, 4, threadIdx.x);
  __syncthreads();
  double mean[3];
  for (int c = 0; c < 3; c++) mean[c] = __ddiv_rn(s_mean[c + 1], s_mean[0]);
  long long i0, i1;
  block_range((long long)im.H * im.W, i0, i1);
  double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (long long i = i0 + threadIdx.x; i < i1; i += STAIN_THREADS) {
    double od[3];
    pixel_od(im, i, s_od, od);
    if (od[0] >= im.beta && od[1] >= im.beta && od[2] >= im.beta) {
      const double d[3] = {__dsub_rn(od[0], mean[0]), __dsub_rn(od[1], mean[1]), __dsub_rn(od[2], mean[2])};
      int k = 0;
      for (int a = 0; a < 3; a++)
        for (int b = a; b < 3; b++, k++) acc[k] = __dadd_rn(acc[k], __dmul_rn(d[a], d[b]));
    }
  }
  for (int k = 0; k < 6; k++) s[k][threadIdx.x] = acc[k];
  block_sum<6>(s);
  if (threadIdx.x < 6) part2[blockIdx.x * 6 + threadIdx.x] = s[threadIdx.x][0];
}

// Eigen-decomposition of the 3x3 covariance by cyclic Jacobi rotations (fp64), eigenpairs sorted ascending.
__device__ void jacobi3(double a[3][3], double w[3], double v[3][3]) {
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) v[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 64; sweep++) {
    if (a[0][1] == 0.0 && a[0][2] == 0.0 && a[1][2] == 0.0) break;
    for (int p = 0; p < 2; p++)
      for (int q = p + 1; q < 3; q++) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        double t = fabs(theta) > 1e150 ? 0.5 / theta : (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; k++) {
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq, a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; k++) {
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk, a[q][k] = s * apk + c * aqk;
        }
        a[p][q] = a[q][p] = 0.0;
        for (int k = 0; k < 3; k++) {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = c * vkp - s * vkq, v[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int o[3] = {0, 1, 2};
  for (int i = 0; i < 3; i++)
    for (int j = i + 1; j < 3; j++)
      if (a[o[j]][o[j]] < a[o[i]][o[i]]) {
        const int x = o[i];
        o[i] = o[j], o[j] = x;
      }
  double vs[3][3];
  for (int k = 0; k < 3; k++) {
    w[k] = a[o[k]][o[k]];
    for (int r = 0; r < 3; r++) vs[r][k] = v[r][o[k]];
  }
  for (int r = 0; r < 3; r++)
    for (int k = 0; k < 3; k++) v[r][k] = vs[r][k];
}

__global__ void k_stain_eig(const double* __restrict__ part1, const double* __restrict__ part2, StainState* st, double alpha) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double n = partial_sum(part1, 4, 0);
  st->n_hat = (long long)n;
  st->valid = n >= 2.0;
  double a[3][3], w[3], v[3][3];
  const double nm1 = n >= 2.0 ? n - 1.0 : 1.0;
  int k = 0;
  for (int i = 0; i < 3; i++)
    for (int j = i; j < 3; j++, k++) a[i][j] = a[j][i] = __ddiv_rn(partial_sum(part2, 6, k), nm1);
  jacobi3(a, w, v);
  for (int r = 0; r < 3; r++) st->E[r][0] = v[r][1], st->E[r][1] = v[r][2];
  set_percentile(st, 0, st->n_hat, alpha / 100.0, 0);
  set_percentile(st, 1, st->n_hat, (100.0 - alpha) / 100.0, 0);
}

__global__ void __launch_bounds__(STAIN_THREADS) k_stain_phi(const StainImage im, const StainState* __restrict__ st,
                                                             unsigned long long* __restrict__ keys) {
  __shared__ double s_od[256];
  fill_od(s_od, im.io);
  __syncthreads();
  double E[3][2];
  for (int r = 0; r < 3; r++) E[r][0] = st->E[r][0], E[r][1] = st->E[r][1];
  const long long n = (long long)im.H * im.W;
  for (long long i = (long long)blockIdx.x * STAIN_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * STAIN_THREADS) {
    double od[3];
    pixel_od(im, i, s_od, od);
    unsigned long long key = kInfKey;
    if (od[0] >= im.beta && od[1] >= im.beta && od[2] >= im.beta) {
      const double t0 = __dadd_rn(__dadd_rn(__dmul_rn(od[0], E[0][0]), __dmul_rn(od[1], E[1][0])), __dmul_rn(od[2], E[2][0]));
      const double t1 = __dadd_rn(__dadd_rn(__dmul_rn(od[0], E[0][1]), __dmul_rn(od[1], E[1][1])), __dmul_rn(od[2], E[2][1]));
      key = key_of(atan2(t1, t0));
    }
    keys[i] = key;
  }
}

// Targets that share (array, prefix) share one histogram: the lowest such target counts, the others read its bins.
__device__ __forceinline__ void target_leaders(const StainState* st, int* lead) {
  for (int t = 0; t < kTargets; t++) {
    lead[t] = t;
    for (int u = 0; u < t; u++)
      if (st->arr[u] == st->arr[t] && st->prefix[u] == st->prefix[t]) {
        lead[t] = u;
        break;
      }
  }
}

__global__ void __launch_bounds__(STAIN_THREADS) k_stain_hist(const unsigned long long* __restrict__ keys_a,
                                                              const unsigned long long* __restrict__ keys_b, long long n,
                                                              const StainState* __restrict__ st, unsigned int* __restrict__ hist,
                                                              int pass) {
  __shared__ unsigned int s_hist[kTargets][256];
  for (int e = threadIdx.x; e < kTargets * 256; e += STAIN_THREADS) (&s_hist[0][0])[e] = 0;
  int lead[kTargets];
  target_leaders(st, lead);
  unsigned long long prefix[kTargets];
  int arr[kTargets];
  bool any_b = false;
  for (int t = 0; t < kTargets; t++) prefix[t] = st->prefix[t], arr[t] = st->arr[t], any_b |= arr[t] == 1;
  const int shift = 56 - 8 * pass;
  const unsigned long long hi_mask = pass == 0 ? 0ull : ~0ull << (shift + 8);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  // every lane of a warp runs the same iterations (the bound is uniform), so the match below sees all 32 lanes
  for (long long base = (long long)blockIdx.x * STAIN_THREADS; base < n; base += (long long)gridDim.x * STAIN_THREADS) {
    const long long i = base + threadIdx.x;
    const bool in = i < n;
    const unsigned long long ka = in ? keys_a[i] : 0ull, kb = in && any_b ? keys_b[i] : 0ull;
#pragma unroll
    for (int t = 0; t < kTargets; t++) {
      if (lead[t] != t) continue;
      const unsigned long long k = arr[t] ? kb : ka;
      const int bin = in && (k & hi_mask) == prefix[t] ? (int)((k >> shift) & 255) : -1;
      const unsigned peers = __match_any_sync(0xffffffffu, bin);
      if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&s_hist[t][bin], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < kTargets * 256; e += STAIN_THREADS) {
    const unsigned c = (&s_hist[0][0])[e];
    if (c) atomicAdd(&hist[e], c);
  }
}

// one block: fix the next byte of every target from the histograms, then clear them for the next pass
__global__ void __launch_bounds__(STAIN_THREADS) k_stain_pick(StainState* st, unsigned int* __restrict__ hist, int pass) {
  __shared__ unsigned int s_hist[kTargets][256];
  __shared__ int s_lead[kTargets];
  for (int e = threadIdx.x; e < kTargets * 256; e += STAIN_THREADS) {
    (&s_hist[0][0])[e] = hist[e];
    hist[e] = 0;
  }
  if (threadIdx.x == 0) target_leaders(st, s_lead);
  __syncthreads();
  if (threadIdx.x >= kTargets) return;
  const int t = threadIdx.x, shift = 56 - 8 * pass;
  const unsigned int* h = s_hist[s_lead[t]];
  unsigned int rank = st->rank[t], below = 0;
  int b = 0;
  for (; b < 255 && below + h[b] <= rank; b++) below += h[b];
  HIPAC_DEV_ASSERT(below + h[b] > rank);
  st->prefix[t] |= (unsigned long long)b << shift;
  st->rank[t] = rank - below;
}

__global__ void k_stain_he(StainState* st, long long n_px) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double min_phi = percentile_of(st, 0), max_phi = percentile_of(st, 1);
  double vmin[3], vmax[3];
  for (int r = 0; r < 3; r++) {
    vmin[r] = __dadd_rn(__dmul_rn(st->E[r][0], cos(min_phi)), __dmul_rn(st->E[r][1], sin(min_phi)));
    vmax[r] = __dadd_rn(__dmul_rn(st->E[r][0], cos(max_phi)), __dmul_rn(st->E[r][1], sin(max_phi)));
  }
  const bool h_first = vmin[0] > vmax[0];
  for (int r = 0; r < 3; r++) {
    st->he[r][0] = h_first ? vmin[r] : vmax[r];
    st->he[r][1] = h_first ? vmax[r] : vmin[r];
  }
  const double det = pinv_fixed(st->he, st->P);
  if (!(det > 0.0)) st->valid = 0;
  // next: the 99th percentiles of C[0] (keys_a) and C[1] (keys_b) over all pixels
  set_percentile(st, 0, n_px, 0.99, 0);
  set_percentile(st, 1, n_px, 0.99, 1);
}

__global__ void __launch_bounds__(STAIN_THREADS) k_stain_conc(const StainImage im, const StainState* __restrict__ st,
                                                              unsigned long long* __restrict__ keys_a,
                                                              unsigned long long* __restrict__ keys_b) {
  __shared__ double s_od[256];
  fill_od(s_od, im.io);
  __syncthreads();
  double P[2][3];
  for (int i = 0; i < 2; i++)
    for (int j = 0; j < 3; j++) P[i][j] = st->P[i][j];
  const long long n = (long long)im.H * im.W;
  for (long long i = (long long)blockIdx.x * STAIN_THREADS + threadIdx.x; i < n; i += (long long)gridDim.x * STAIN_THREADS) {
    double od[3];
    pixel_od(im, i, s_od, od);
    const double c0 = __dadd_rn(__dadd_rn(__dmul_rn(P[0][0], od[0]), __dmul_rn(P[0][1], od[1])), __dmul_rn(P[0][2], od[2]));
    const double c1 = __dadd_rn(__dadd_rn(__dmul_rn(P[1][0], od[0]), __dmul_rn(P[1][1], od[1])), __dmul_rn(P[1][2], od[2]));
    keys_a[i] = key_of(c0);
    keys_b[i] = key_of(c1);
  }
}

__global__ void k_stain_finish(const StainState* __restrict__ st, double* __restrict__ out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double max_c[2] = {percentile_of(st, 0), percentile_of(st, 1)};
  bool ok = st->valid != 0;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 2; c++) {
      out[r * 2 + c] = st->he[r][c];
      ok &= isfinite(st->he[r][c]);
    }
  for (int c = 0; c < 2; c++) {
    out[6 + c] = max_c[c];
    ok &= isfinite(max_c[c]) && max_c[c] > 0.0;
  }
  out[8] = ok ? 1.0 : 0.0;
  out[9] = (double)st->n_hat;
  for (int k = 10; k < HIPAC_STAIN_BLOCK_DOUBLES; k++) out[k] = 0.0;
}

// ------------------------------------------------------------------------------------------
// normaliser: parameter block from a source and a target stain block
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(STAIN_THREADS) k_stain_normalizer(const double* __restrict__ src, const double* __restrict__ target,
                                                                    int io, double* __restrict__ params) {
  fill_od(params + 11, io);
  if (threadIdx.x != 0) return;
  double he[3][2], he_ref[3][2], P[2][3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 2; c++) he[r][c] = src[r * 2 + c], he_ref[r][c] = target ? target[r * 2 + c] : kHeRef[r][c];
  const double max_c_ref[2] = {target ? target[6] : kMaxCRef[0], target ? target[7] : kMaxCRef[1]};
  bool ok = src[8] != 0.0 && (!target || target[8] != 0.0);
  const double det = pinv_fixed(he, P);
  ok &= det > 0.0;
  const double s[2] = {__ddiv_rn(max_c_ref[0], src[6]), __ddiv_rn(max_c_ref[1], src[7])};
  for (int c = 0; c < 3; c++)
    for (int j = 0; j < 3; j++) {
      const double m = __dadd_rn(__dmul_rn(__dmul_rn(he_ref[c][0], s[0]), P[0][j]), __dmul_rn(__dmul_rn(he_ref[c][1], s[1]), P[1][j]));
      params[2 + c * 3 + j] = m;
      ok &= isfinite(m);
    }
  params[0] = ok ? 1.0 : 0.0;
  params[1] = (double)io;
}

// ------------------------------------------------------------------------------------------
// apply: uint8 [n][224][224][3] -> normalised uint8 and / or the bf16 batch
// ------------------------------------------------------------------------------------------
struct StainApply {
  const uint8_t* in;       // may equal out_u8 (every thread reads its pixels before writing them)
  uint8_t* out_u8;         // or null
  uint16_t* batch;         // bf16 bits, or null (LAYOUT 0)
  const double* params;
  const int* n_dev;        // device-count mode, or null
  int n_base, n_img;
  uint16_t lut[768];       // [v][c] bf16 bits of ToTensor/Normalize
};

__device__ __forceinline__ uint32_t stain_channel(double y, const double* od, float io) {
  const float g = io * __expf(-(float)y);   // a guess, confirmed below against the exact fp64 thresholds
  int k = g >= 255.0f ? 255 : (g > 0.0f ? (int)g : 0);
  while (k < 255 && y <= od[k]) k++;
  while (k > 0 && y > od[k - 1]) k--;
  return (uint32_t)k;
}

// one thread = 2 rows x 4 pixels (two S2D16 blocks): 12-byte input runs per row, 4-byte aligned
template <int LAYOUT>
__global__ void __launch_bounds__(STAIN_THREADS) k_stain_apply(const __grid_constant__ StainApply p) {
  __shared__ double s_a[3][3][256];
  __shared__ double s_od[256];
  __shared__ uint16_t s_lut[768];
  const bool valid = p.params[0] != 0.0;
  const float io = (float)p.params[1];
  for (int e = threadIdx.x; e < 256; e += STAIN_THREADS) s_od[e] = p.params[11 + e];
  for (int e = threadIdx.x; e < 9 * 256; e += STAIN_THREADS) (&s_a[0][0][0])[e] = __dmul_rn(p.params[2 + e / 256], p.params[11 + e % 256]);
  if (LAYOUT) for (int e = threadIdx.x; e < 768; e += STAIN_THREADS) s_lut[e] = p.lut[e];
  __syncthreads();
  int n = p.n_img;
  if (p.n_dev) n = max(0, min(n, __ldg(p.n_dev) - p.n_base));
  const int64_t total = (int64_t)n * 112 * 56;
  for (int64_t t = (int64_t)blockIdx.x * STAIN_THREADS + threadIdx.x; t < total; t += (int64_t)gridDim.x * STAIN_THREADS) {
    const int u = (int)(t % 56), Y = (int)((t / 56) % 112);
    const int64_t img = t / (112 * 56);
    HIPAC_DEV_ASSERT(img < p.n_img && Y < 112 && u < 56);
    uint32_t w[2][3];
#pragma unroll
    for (int sy = 0; sy < 2; sy++) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(p.in + ((img * 224 + 2 * Y + sy) * 224 + 4 * u) * 3);
#pragma unroll
      for (int k = 0; k < 3; k++) w[sy][k] = src[k];
    }
    if (valid) {
#pragma unroll
      for (int sy = 0; sy < 2; sy++) {
        uint32_t o[3] = {0u, 0u, 0u};
#pragma unroll
        for (int x = 0; x < 4; x++) {
          const int b0 = 3 * x;
          const uint32_t r = (w[sy][b0 >> 2] >> (8 * (b0 & 3))) & 255, g = (w[sy][(b0 + 1) >> 2] >> (8 * ((b0 + 1) & 3))) & 255,
                         b = (w[sy][(b0 + 2) >> 2] >> (8 * ((b0 + 2) & 3))) & 255;
#pragma unroll
          for (int c = 0; c < 3; c++) {
            const double y = __dadd_rn(__dadd_rn(s_a[c][0][r], s_a[c][1][g]), s_a[c][2][b]);
            const int bc = b0 + c;
            o[bc >> 2] |= stain_channel(y, s_od, io) << (8 * (bc & 3));
          }
        }
#pragma unroll
        for (int k = 0; k < 3; k++) w[sy][k] = o[k];
      }
    }
    if (p.out_u8) {
#pragma unroll
      for (int sy = 0; sy < 2; sy++) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(p.out_u8 + ((img * 224 + 2 * Y + sy) * 224 + 4 * u) * 3);
#pragma unroll
        for (int k = 0; k < 3; k++) dst[k] = w[sy][k];
      }
    }
    if (LAYOUT == HIPAC_LAYOUT_NHWC3_BF16) {
#pragma unroll
      for (int sy = 0; sy < 2; sy++) {
        uint32_t h[6];
#pragma unroll
        for (int e = 0; e < 6; e++) {
          const int b0 = 2 * e, b1 = 2 * e + 1;
          h[e] = (uint32_t)s_lut[((w[sy][b0 >> 2] >> (8 * (b0 & 3))) & 255) * 3 + b0 % 3] |
                 ((uint32_t)s_lut[((w[sy][b1 >> 2] >> (8 * (b1 & 3))) & 255) * 3 + b1 % 3] << 16);
        }
        uint2* dst = reinterpret_cast<uint2*>(p.batch + ((img * 224 + 2 * Y + sy) * 224 + 4 * u) * 3);   // 24 bytes, 8-aligned
#pragma unroll
        for (int k = 0; k < 3; k++) dst[k] = make_uint2(h[2 * k], h[2 * k + 1]);
      }
    } else if (LAYOUT == HIPAC_LAYOUT_S2D16_BF16) {
      // block X = 2u + xb: channel (sy * 2 + sx) * 3 + c = pixel (2Y + sy, 4u + 2xb + sx)
      uint4* row = reinterpret_cast<uint4*>(p.batch + (img * 112 + Y) * HIPAC_S2D16_WIDTH * 16);
#pragma unroll
      for (int xb = 0; xb < 2; xb++) {
        uint32_t h[8];
#pragma unroll
        for (int e = 0; e < 6; e++) {
          uint32_t pair[2];
#pragma unroll
          for (int z = 0; z < 2; z++) {
            const int ch = 2 * e + z, sy = ch / 6, sx = (ch / 3) & 1, c = ch % 3;
            const int bi = (2 * xb + sx) * 3 + c;
            pair[z] = s_lut[((w[sy][bi >> 2] >> (8 * (bi & 3))) & 255) * 3 + c];
          }
          h[e] = pair[0] | (pair[1] << 16);
        }
        h[6] = h[7] = 0u;
        uint4* dst = row + (2 * u + xb + 2) * 2;
        dst[0] = make_uint4(h[0], h[1], h[2], h[3]);
        dst[1] = make_uint4(h[4], h[5], h[6], h[7]);
      }
      const uint4 z = make_uint4(0u, 0u, 0u, 0u);
      if (u == 0) row[0] = row[1] = row[2] = row[3] = z;                   // columns X = -2, -1
      if (u == 55) row[(112 + 2) * 2] = row[(112 + 2) * 2 + 1] = z;        // column X = 112
    }
  }
}

}  // namespace hipac

// ==========================================================================================
// C ABI
// ==========================================================================================
using namespace hipac;

namespace {
struct StainWs {
  StainState* st;
  double* part1;
  double* part2;
  unsigned int* hist;
  unsigned long long* keys_a;
  unsigned long long* keys_b;
  size_t bytes;
};

StainWs stain_ws(void* base, int H, int W) {
  StainWs w;
  size_t off = 0;
  uint8_t* b = reinterpret_cast<uint8_t*>(base);
  auto carve = [&](size_t bytes) {
    uint8_t* r = b ? b + off : nullptr;
    off += align_up(bytes, 256);
    return r;
  };
  const size_t n = (size_t)H * W;
  w.st = reinterpret_cast<StainState*>(carve(sizeof(StainState)));
  w.part1 = reinterpret_cast<double*>(carve(STAIN_RED_BLOCKS * 4 * sizeof(double)));
  w.part2 = reinterpret_cast<double*>(carve(STAIN_RED_BLOCKS * 6 * sizeof(double)));
  w.hist = reinterpret_cast<unsigned int*>(carve(kTargets * 256 * sizeof(unsigned int)));
  w.keys_a = reinterpret_cast<unsigned long long*>(carve(n * 8));
  w.keys_b = reinterpret_cast<unsigned long long*>(carve(n * 8));
  w.bytes = off;
  return w;
}

int stain_select(const StainWs& w, long long n, int grid, cudaStream_t stream) {
  for (int pass = 0; pass < 8; pass++) {
    {
      ProfileScope ps("stain_hist", stream, (double)n * 16);
      k_stain_hist<<<grid, STAIN_THREADS, 0, stream>>>(w.keys_a, w.keys_b, n, w.st, w.hist, pass);
    }
    count_launch(1);
    {
      ProfileScope ps("stain_pick", stream, 0.0);
      k_stain_pick<<<1, STAIN_THREADS, 0, stream>>>(w.st, w.hist, pass);
    }
    count_launch(1);
  }
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace

extern "C" size_t hipac_stain_workspace_bytes(int H, int W) {
  if (H <= 0 || W <= 0) {
    set_error("invalid argument: empty image");
    return 0;
  }
  if ((int64_t)H * W >= ((int64_t)1 << 31)) {
    set_error("invalid argument: image has 2^31 pixels or more");
    return 0;
  }
  return stain_ws(nullptr, H, W).bytes;
}

extern "C" int hipac_stain_estimate(const uint8_t* d_rgb, int H, int W, int64_t pitch, int Io, double alpha, double beta,
                                    double* d_stain, void* d_ws, size_t ws_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  HIPAC_REQUIRE(d_rgb && d_stain && d_ws, "null pointer");
  HIPAC_REQUIRE(H > 0 && W > 0, "empty image");
  HIPAC_REQUIRE((int64_t)H * W < ((int64_t)1 << 31), "image has 2^31 pixels or more");
  HIPAC_REQUIRE(pitch >= (int64_t)W * 3, "pitch smaller than a row");
  HIPAC_REQUIRE(Io >= 1 && Io <= 255, "Io must be in 1..255");
  HIPAC_REQUIRE(alpha > 0.0 && alpha < 50.0, "alpha must be in (0, 50)");
  HIPAC_REQUIRE(beta >= 0.0 && beta < HUGE_VAL, "beta must be finite and >= 0");
  HIPAC_REQUIRE(((uintptr_t)d_ws & 255) == 0, "workspace must be 256-byte aligned");
  HIPAC_REQUIRE(ws_bytes >= hipac_stain_workspace_bytes(H, W), "workspace too small");
  const StainWs w = stain_ws(d_ws, H, W);
  const StainImage im{d_rgb, H, W, pitch, Io, beta};
  const long long n = (long long)H * W;
  int sms = 0;
  if (int e = device_sm_count(&sms)) return e;
  const int grid = (int)std::min<long long>((n + STAIN_THREADS - 1) / STAIN_THREADS, (long long)sms * 8);
  HIPAC_CHECK_CUDA(cudaMemsetAsync(w.hist, 0, kTargets * 256 * sizeof(unsigned int), stream));
  {
    ProfileScope ps("stain_sums", stream, (double)n * 3);
    k_stain_sums<<<STAIN_RED_BLOCKS, STAIN_THREADS, 0, stream>>>(im, w.part1);
  }
  count_launch(1);
  {
    ProfileScope ps("stain_cov", stream, (double)n * 3);
    k_stain_cov<<<STAIN_RED_BLOCKS, STAIN_THREADS, 0, stream>>>(im, w.part1, w.part2);
  }
  count_launch(1);
  {
    ProfileScope ps("stain_eig", stream, 0.0);
    k_stain_eig<<<1, 32, 0, stream>>>(w.part1, w.part2, w.st, alpha);
  }
  count_launch(1);
  {
    ProfileScope ps("stain_phi", stream, (double)n * 11);
    k_stain_phi<<<grid, STAIN_THREADS, 0, stream>>>(im, w.st, w.keys_a);
  }
  count_launch(1);
  if (int e = stain_select(w, n, grid, stream)) return e;
  {
    ProfileScope ps("stain_he", stream, 0.0);
    k_stain_he<<<1, 32, 0, stream>>>(w.st, n);
  }
  count_launch(1);
  {
    ProfileScope ps("stain_conc", stream, (double)n * 19);
    k_stain_conc<<<grid, STAIN_THREADS, 0, stream>>>(im, w.st, w.keys_a, w.keys_b);
  }
  count_launch(1);
  if (int e = stain_select(w, n, grid, stream)) return e;
  {
    ProfileScope ps("stain_finish", stream, 0.0);
    k_stain_finish<<<1, 32, 0, stream>>>(w.st, d_stain);
  }
  count_launch(1);
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int hipac_stain_normalizer(const double* d_src, const double* d_target, int Io, double* d_params, void* stream_) {
  HIPAC_REQUIRE(d_src && d_params, "null pointer");
  HIPAC_REQUIRE(Io >= 1 && Io <= 255, "Io must be in 1..255");
  cudaStream_t stream = (cudaStream_t)stream_;
  {
    ProfileScope ps("stain_normalizer", stream, 0.0);
    k_stain_normalizer<<<1, STAIN_THREADS, 0, stream>>>(d_src, d_target, Io, d_params);
  }
  count_launch(1);
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}

static bool overlap(uintptr_t a, size_t na, uintptr_t b, size_t nb) { return na && nb && a < b + nb && b < a + na; }

extern "C" int hipac_stain_apply(const uint8_t* d_in, int n_patches, const int32_t* d_count, int n_base, const double* d_params,
                                 uint8_t* d_out_u8, void* d_batch, int layout, void* stream_) {
  HIPAC_REQUIRE(d_in && d_params, "null pointer");
  HIPAC_REQUIRE(n_patches >= 0, "negative n_patches");
  HIPAC_REQUIRE(n_base >= 0, "n_base must be non-negative");
  HIPAC_REQUIRE(layout == 0 || layout == HIPAC_LAYOUT_NHWC3_BF16 || layout == HIPAC_LAYOUT_S2D16_BF16, "unknown batch layout");
  HIPAC_REQUIRE((layout != 0) == (d_batch != nullptr), "d_batch needs a layout and a layout needs d_batch");
  HIPAC_REQUIRE(d_out_u8 || d_batch, "no output");
  HIPAC_REQUIRE(((uintptr_t)d_in & 15) == 0 && ((uintptr_t)d_out_u8 & 15) == 0 && ((uintptr_t)d_batch & 15) == 0,
                "buffers must be 16-byte aligned");
  const size_t u8_bytes = (size_t)n_patches * 224 * 224 * 3;
  const size_t bf_bytes = (size_t)n_patches * (layout == HIPAC_LAYOUT_S2D16_BF16 ? (size_t)112 * HIPAC_S2D16_WIDTH * 32 : (size_t)224 * 224 * 6);
  const uintptr_t in = (uintptr_t)d_in, o8 = (uintptr_t)d_out_u8, ob = (uintptr_t)d_batch;
  HIPAC_REQUIRE(!d_out_u8 || o8 == in || !overlap(in, u8_bytes, o8, u8_bytes), "d_out_u8 partially overlaps d_in");
  HIPAC_REQUIRE(!d_batch || !overlap(in, u8_bytes, ob, bf_bytes), "d_batch overlaps d_in");
  HIPAC_REQUIRE(!d_batch || !d_out_u8 || !overlap(o8, u8_bytes, ob, bf_bytes), "d_batch overlaps d_out_u8");
  if (n_patches == 0) return 0;
  cudaStream_t stream = (cudaStream_t)stream_;
  int sms = 0;
  if (int e = device_sm_count(&sms)) return e;
  static StainApply proto = [] {
    StainApply a{};
    host_normalize_lut_bf16(a.lut);
    return a;
  }();
  StainApply p = proto;
  p.in = d_in, p.out_u8 = d_out_u8, p.batch = reinterpret_cast<uint16_t*>(d_batch), p.params = d_params;
  p.n_dev = d_count, p.n_base = n_base, p.n_img = n_patches;
  const int64_t units = (int64_t)n_patches * 112 * 56;
  const int grid = (int)std::min<int64_t>((units + STAIN_THREADS - 1) / STAIN_THREADS, (int64_t)sms * STAIN_APPLY_CTAS_PER_SM);
  {
    ProfileScope ps("stain_apply", stream, (double)u8_bytes * (d_out_u8 ? 2 : 1) + (double)(d_batch ? bf_bytes : 0));
    if (layout == HIPAC_LAYOUT_S2D16_BF16) k_stain_apply<HIPAC_LAYOUT_S2D16_BF16><<<grid, STAIN_THREADS, 0, stream>>>(p);
    else if (layout == HIPAC_LAYOUT_NHWC3_BF16) k_stain_apply<HIPAC_LAYOUT_NHWC3_BF16><<<grid, STAIN_THREADS, 0, stream>>>(p);
    else k_stain_apply<0><<<grid, STAIN_THREADS, 0, stream>>>(p);
  }
  count_launch(1);
  HIPAC_CHECK_CUDA(cudaGetLastError());
  return 0;
}
