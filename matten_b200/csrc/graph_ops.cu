// Edge geometry + index bookkeeping kernels (rows a1-a4 of SURVEY.md section 8).
#include "common.cuh"
#include "generated/cg_gen.cuh"
#include "soft_one_hot.cuh"

namespace mt {

// =========================================================================
// a1: edge vectors / lengths            reference src/matten/nn/_nequip.py:214-268
// =========================================================================
template <typename T>
__global__ void __launch_bounds__(256) edge_vectors_kernel(
    const T* __restrict__ pos, const int64_t* __restrict__ ei, const T* __restrict__ shift,
    const T* __restrict__ cell, const int64_t* __restrict__ batch, int64_t N, int64_t E, int64_t B,
    T* __restrict__ vec, T* __restrict__ len, int32_t* __restrict__ err_flag) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  int64_t i = ei[e], j = ei[E + e];
  if (i < 0 || i >= N || j < 0 || j >= N) {
    if (err_flag) atomicOr(err_flag, MT_FLAG_BAD_INDEX);
    i = 0;
    j = 0;
  }
  T v0 = pos[j * 3 + 0] - pos[i * 3 + 0];
  T v1 = pos[j * 3 + 1] - pos[i * 3 + 1];
  T v2 = pos[j * 3 + 2] - pos[i * 3 + 2];
  if (cell != nullptr) {
    int64_t g = 0;
    if (B > 1) {
      g = batch[i];
      if (g < 0 || g >= B) {
        if (err_flag) atomicOr(err_flag, MT_FLAG_BAD_INDEX);
        g = 0;
      }
    }
    const T* c = cell + g * 9;
    T s0 = shift[e * 3 + 0], s1 = shift[e * 3 + 1], s2 = shift[e * 3 + 2];
    // einsum("ni,nij->nj"): rows of the cell are the lattice vectors
    v0 += s0 * c[0] + s1 * c[3] + s2 * c[6];
    v1 += s0 * c[1] + s1 * c[4] + s2 * c[7];
    v2 += s0 * c[2] + s1 * c[5] + s2 * c[8];
  }
  if (vec) {
    vec[e * 3 + 0] = v0;
    vec[e * 3 + 1] = v1;
    vec[e * 3 + 2] = v2;
  }
  if (len) len[e] = sqrt(v0 * v0 + v1 * v1 + v2 * v2);
}

// =========================================================================
// a2: spherical harmonics               reference src/matten/nn/_nequip.py:167-176
// =========================================================================
template <typename T, int LMAXV>
__global__ void __launch_bounds__(256) edge_sh_kernel(const T* __restrict__ vec, int64_t E, int normalize,
                                                      T* __restrict__ out) {
  constexpr int D = (LMAXV + 1) * (LMAXV + 1);
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  T x = vec[e * 3 + 0], y = vec[e * 3 + 1], z = vec[e * 3 + 2];
  if (normalize) {
    // torch.nn.functional.normalize: v / max(|v|, 1e-12)
    T n = sqrt(x * x + y * y + z * z);
    n = n > T(1e-12) ? n : T(1e-12);
    x /= n;
    y /= n;
    z /= n;
  }
  T sh[D];
  sh_component<LMAXV, T>(x, y, z, sh);
  T* o = out + e * D;
#pragma unroll
  for (int k = 0; k < D; ++k) o[k] = sh[k];
}

// =========================================================================
// a3 / a3': radial basis                reference src/matten/nn/embedding.py:185-203,
//                                        src/matten/nn/_nequip.py:43-126
// =========================================================================
template <typename T>
__global__ void __launch_bounds__(256) edge_radial_kernel(const T* __restrict__ len, int64_t E, int mode,
                                                          int nb, T start, T end, int cutoff, T poly_p,
                                                          const T* __restrict__ bessel_w,
                                                          T* __restrict__ out) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= E * nb) return;
  int64_t e = t / nb;
  int k = (int)(t - e * nb);
  const T pi = T(3.14159265358979323846);
  T r = len[e];
  T v;
  if (mode == 0) {
    T x = r - start;
    T c = end - start;
    T root = T(k + 1) * pi;
    v = sqrt(T(2) / c) * sin(root * x / c) / x;
    if (cutoff) {
      // the reference multiplies by the two boolean masks, so r == 0 stays NaN (0/0 * 0)
      v = v * (((x / c) < T(1)) ? T(1) : T(0)) * ((T(0) < x) ? T(1) : T(0));
    }
    v *= sqrt(T(nb));
  } else if (mode <= 2) {
    T w = bessel_w ? bessel_w[k] : T(k + 1) * pi;
    // mode 2: derivative of the mode-1 value with respect to the frequency w_k (trainable BesselBasis)
    T basis = mode == 2 ? (T(2) / end) * (cos(w * r / end) / end) : (T(2) / end) * (sin(w * r / end) / r);
    T u = r / end;
    T p = poly_p;
    T env = T(1) - ((p + T(1)) * (p + T(2)) / T(2)) * pow(u, p) + p * (p + T(2)) * pow(u, p + T(1)) -
            (p * (p + T(1)) / T(2)) * pow(u, p + T(2));
    env *= (r < end) ? T(1) : T(0);
    v = basis * env;
  } else {
    v = soft_one_hot<T, false>(mode, k, nb, r, start, end, cutoff);
  }
  out[t] = v;
}

// =========================================================================
// backward of a1 - a3 (first derivatives; reference autograd through the same lines)
// =========================================================================
template <typename T, int LMAXV>
__global__ void __launch_bounds__(256) edge_sh_bwd_kernel(const T* __restrict__ vec, const T* __restrict__ gsh,
                                                          int64_t E, int normalize, T* __restrict__ gvec) {
  constexpr int D = (LMAXV + 1) * (LMAXV + 1);
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  T x = vec[e * 3 + 0], y = vec[e * 3 + 1], z = vec[e * 3 + 2];
  T nr = T(1), n = T(1);
  if (normalize) {
    nr = sqrt(x * x + y * y + z * z);
    n = nr > T(1e-12) ? nr : T(1e-12);
    x /= n;
    y /= n;
    z /= n;
  }
  T g[D], gu[3];
#pragma unroll
  for (int k = 0; k < D; ++k) g[k] = gsh[e * D + k];
  sh_component_vjp<LMAXV, T>(x, y, z, g, gu);
  if (normalize) {
    // d (v / max(|v|, eps)) / d v: (I - u u^T) / |v| above eps, I / eps below (the clamp has zero derivative)
    const T ug = nr > T(1e-12) ? x * gu[0] + y * gu[1] + z * gu[2] : T(0);
    gu[0] = (gu[0] - x * ug) / n;
    gu[1] = (gu[1] - y * ug) / n;
    gu[2] = (gu[2] - z * ug) / n;
  }
  gvec[e * 3 + 0] = gu[0];
  gvec[e * 3 + 1] = gu[1];
  gvec[e * 3 + 2] = gu[2];
}

template <typename T>
__global__ void __launch_bounds__(256) edge_radial_bwd_kernel(const T* __restrict__ len, const T* __restrict__ g,
                                                              int64_t E, int mode, int nb, T start, T end, int cutoff,
                                                              T poly_p, const T* __restrict__ bessel_w,
                                                              T* __restrict__ glen) {
  int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (e >= E) return;
  const T pi = T(3.14159265358979323846);
  const T r = len[e];
  const T* gr = g + e * nb;
  T acc = T(0);
  if (mode == 0) {
    // d/dx [sqrt(2/c) sin(a x) / x] = sqrt(2/c) (a x cos(a x) - sin(a x)) / x^2, times the (constant) masks, sqrt(n)
    const T x = r - start, c = end - start;
    const T mask = cutoff ? ((((x / c) < T(1)) ? T(1) : T(0)) * ((T(0) < x) ? T(1) : T(0))) : T(1);
    const T s = sqrt(T(2) / c) * mask * sqrt(T(nb));
    for (int k = 0; k < nb; ++k) {
      const T a = T(k + 1) * pi / c;
      acc = fma(gr[k], s * (a * x * cos(a * x) - sin(a * x)) / (x * x), acc);
    }
  } else if (mode == 1) {
    const T u = r / end, p = poly_p;
    const T env = T(1) - ((p + T(1)) * (p + T(2)) / T(2)) * pow(u, p) + p * (p + T(2)) * pow(u, p + T(1)) -
                  (p * (p + T(1)) / T(2)) * pow(u, p + T(2));
    const T denv = (-((p + T(1)) * (p + T(2)) / T(2)) * p * pow(u, p - T(1)) +
                    p * (p + T(2)) * (p + T(1)) * pow(u, p) - (p * (p + T(1)) / T(2)) * (p + T(2)) * pow(u, p + T(1))) /
                   end;
    const T inside = (r < end) ? T(1) : T(0);
    for (int k = 0; k < nb; ++k) {
      const T w = bessel_w ? bessel_w[k] : T(k + 1) * pi;
      const T basis = (T(2) / end) * (sin(w * r / end) / r);
      const T dbasis = (T(2) / end) * ((w / end) * r * cos(w * r / end) - sin(w * r / end)) / (r * r);
      acc = fma(gr[k], (dbasis * env + basis * denv) * inside, acc);
    }
  } else {
    for (int k = 0; k < nb; ++k) acc = fma(gr[k], soft_one_hot<T, true>(mode, k, nb, r, start, end, cutoff), acc);
  }
  glen[e] = acc;
}

// dv of every edge in receiver-sorted order (position i holds edge perm[i]), and shift (x) dv for the cell
template <typename T>
__global__ void __launch_bounds__(256) edge_dv_kernel(const T* __restrict__ vec, const T* __restrict__ gvec,
                                                      const T* __restrict__ glen, const T* __restrict__ shift,
                                                      const int32_t* __restrict__ perm, int64_t E,
                                                      T* __restrict__ dvs, T* __restrict__ sdv) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= E) return;
  const int64_t e = perm[i];
  T d[3] = {T(0), T(0), T(0)};
  if (gvec) {
    d[0] = gvec[e * 3 + 0];
    d[1] = gvec[e * 3 + 1];
    d[2] = gvec[e * 3 + 2];
  }
  if (glen) {
    const T v0 = vec[e * 3 + 0], v1 = vec[e * 3 + 1], v2 = vec[e * 3 + 2];
    const T n = sqrt(v0 * v0 + v1 * v1 + v2 * v2);
    if (n > T(0)) {
      const T s = glen[e] / n;
      d[0] = fma(s, v0, d[0]);
      d[1] = fma(s, v1, d[1]);
      d[2] = fma(s, v2, d[2]);
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) dvs[i * 3 + c] = d[c];
  if (sdv) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const T sa = shift[e * 3 + a];
#pragma unroll
      for (int b = 0; b < 3; ++b) sdv[i * 9 + a * 3 + b] = sa * d[b];
    }
  }
}

// grad_pos[n] = (sum of dv over the edges received by n) - (sum over the edges sent by n), both in CSR order
template <typename T>
__global__ void __launch_bounds__(256) pos_grad_kernel(const T* __restrict__ dvs, const int32_t* __restrict__ rowptr,
                                                       const int32_t* __restrict__ sptr,
                                                       const int32_t* __restrict__ sperm, int64_t N,
                                                       T* __restrict__ gpos) {
  int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (n >= N) return;
  T r[3] = {T(0), T(0), T(0)}, s[3] = {T(0), T(0), T(0)};
  for (int32_t i = rowptr[n]; i < rowptr[n + 1]; ++i)
#pragma unroll
    for (int c = 0; c < 3; ++c) r[c] += dvs[(int64_t)i * 3 + c];
  for (int32_t j = sptr[n]; j < sptr[n + 1]; ++j) {
    const int64_t i = sperm[j];
#pragma unroll
    for (int c = 0; c < 3; ++c) s[c] += dvs[i * 3 + c];
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) gpos[n * 3 + c] = r[c] - s[c];
}

// segment bounds of every graph in the sender CSR: the edges sent by nodes graph_ptr[g] .. graph_ptr[g+1]
__global__ void __launch_bounds__(256) graph_edge_ptr_kernel(const int32_t* __restrict__ sptr,
                                                             const int32_t* __restrict__ graph_ptr, int64_t B,
                                                             int64_t N, int32_t* __restrict__ out) {
  int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (g > B) return;
  out[g] = sptr[graph_ptr ? graph_ptr[g] : (g == 0 ? 0 : N)];
}

// =========================================================================
// exclusive scan (int32), multi-level
// =========================================================================
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__global__ void __launch_bounds__(kScanThreads) scan_tile_kernel(int32_t* __restrict__ data, int64_t n,
                                                                 int32_t* __restrict__ tile_sums) {
  __shared__ int32_t warp_sums[kScanThreads / 32];
  int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  int32_t v[kScanItems];
  int32_t tsum = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    v[i] = (base + i < n) ? data[base + i] : 0;
    tsum += v[i];
  }
  // inclusive warp scan of thread sums
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int32_t inc = tsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  int32_t woff = 0;
  for (int w = 0; w < warp; ++w) woff += warp_sums[w];
  int32_t excl = woff + inc - tsum;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < n) data[base + i] = excl;
    excl += v[i];
  }
  if (threadIdx.x == kScanThreads - 1 && tile_sums) tile_sums[blockIdx.x] = woff + inc;
}

__global__ void __launch_bounds__(kScanThreads) scan_add_kernel(int32_t* __restrict__ data, int64_t n,
                                                                const int32_t* __restrict__ tile_offs) {
  int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  int32_t off = tile_offs[blockIdx.x];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < n) data[base + i] += off;
}

static size_t scan_tmp_elems(int64_t n) {
  size_t total = 0;
  while (n > kScanTile) {
    n = ceil_div<int64_t>(n, kScanTile);
    total += (size_t)n;
  }
  return total + 1;
}

// in-place exclusive scan of data[0..n)
static int exclusive_scan_i32(int32_t* data, int64_t n, int32_t* tmp, cudaStream_t st) {
  if (n <= 0) return MT_OK;
  int64_t nb = ceil_div<int64_t>(n, kScanTile);
  if (nb == 1) {
    scan_tile_kernel<<<1, kScanThreads, 0, st>>>(data, n, nullptr);
    MT_LAUNCH_OK();
    return MT_OK;
  }
  scan_tile_kernel<<<(unsigned)nb, kScanThreads, 0, st>>>(data, n, tmp);
  MT_LAUNCH_OK();
  int rc = exclusive_scan_i32(tmp, nb, tmp + nb, st);
  if (rc != MT_OK) return rc;
  scan_add_kernel<<<(unsigned)nb, kScanThreads, 0, st>>>(data, n, tmp);
  MT_LAUNCH_OK();
  return MT_OK;
}

// =========================================================================
// stable LSD radix sort of (key, index) pairs, 8 bits per pass
// =========================================================================
constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortRounds = 8;                                  // 32-element rounds per warp
constexpr int kSortTile = kSortThreads * kSortRounds;           // 2048 elements per block

__global__ void __launch_bounds__(256) keys_init_kernel(const int64_t* __restrict__ keys, int64_t E,
                                                        int64_t num_keys, int32_t* __restrict__ k32,
                                                        int32_t* __restrict__ idx,
                                                        int32_t* __restrict__ err_flag) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= E) return;
  int64_t k = keys[i];
  if (k < 0 || k >= num_keys) {
    if (err_flag) atomicOr(err_flag, MT_FLAG_BAD_INDEX);
    k = 0;
  }
  k32[i] = (int32_t)k;
  if (idx) idx[i] = (int32_t)i;
}

// element (warp w, round r, lane l) of block b is at  b*tile + w*(32*rounds) + r*32 + l
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const int32_t* __restrict__ keys,
                                                                  int64_t E, int shift,
                                                                  int32_t* __restrict__ hist,
                                                                  int nblocks) {
  __shared__ int32_t cnt[256];
  cnt[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * kSortTile;
  for (int r = 0; r < kSortRounds; ++r) {
    int64_t i = base + (int64_t)r * kSortThreads + threadIdx.x;
    if (i < E) atomicAdd(&cnt[(keys[i] >> shift) & 255], 1);
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * nblocks + blockIdx.x] = cnt[threadIdx.x];
}

__global__ void __launch_bounds__(kSortThreads) radix_scatter_kernel(
    const int32_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in, int64_t E, int shift,
    const int32_t* __restrict__ hist_scanned, int nblocks, int32_t* __restrict__ keys_out,
    int32_t* __restrict__ vals_out) {
  __shared__ int32_t wcnt[kSortWarps][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < kSortWarps * 256; i += kSortThreads) (&wcnt[0][0])[i] = 0;
  __syncthreads();
  const int64_t wbase = (int64_t)blockIdx.x * kSortTile + (int64_t)warp * (32 * kSortRounds);
  int32_t k[kSortRounds], v[kSortRounds];
  // phase 1: per-warp digit counts
#pragma unroll
  for (int r = 0; r < kSortRounds; ++r) {
    int64_t i = wbase + r * 32 + lane;
    bool valid = i < E;
    k[r] = valid ? keys_in[i] : 0;
    v[r] = valid ? vals_in[i] : 0;
    int d = valid ? ((k[r] >> shift) & 255) : 256;  // 256: invalid lanes match among themselves
    unsigned m = __match_any_sync(0xffffffffu, d);
    if (valid && (__ffs(m) - 1) == lane) wcnt[warp][d] += __popc(m);
    __syncwarp();
  }
  __syncthreads();
  // exclusive prefix over warps + global offset of (digit, block)
  {
    int d = threadIdx.x;  // 256 threads == 256 digits
    int32_t run = hist_scanned[(int64_t)d * nblocks + blockIdx.x];
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) {
      int32_t c = wcnt[w][d];
      wcnt[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
  // phase 2: stable placement
#pragma unroll
  for (int r = 0; r < kSortRounds; ++r) {
    int64_t i = wbase + r * 32 + lane;
    bool valid = i < E;
    int d = valid ? ((k[r] >> shift) & 255) : 256;
    unsigned m = __match_any_sync(0xffffffffu, d);
    int rank = __popc(m & ((1u << lane) - 1u));
    if (valid) {
      int32_t pos = wcnt[warp][d] + rank;
      keys_out[pos] = k[r];
      vals_out[pos] = v[r];
    }
    __syncwarp();
    if (valid && (__ffs(m) - 1) == lane) wcnt[warp][d] += __popc(m);
    __syncwarp();
  }
}

// rowptr from sorted keys: rowptr[k] = first position whose key >= k
__global__ void __launch_bounds__(256) rowptr_from_sorted_kernel(const int32_t* __restrict__ skeys,
                                                                 int64_t E, int64_t num_keys,
                                                                 int32_t* __restrict__ rowptr) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i > E) return;
  int64_t lo = (i == 0) ? -1 : skeys[i - 1];
  int64_t hi = (i == E) ? num_keys : skeys[i];
  for (int64_t k = lo + 1; k <= hi; ++k) rowptr[k] = (int32_t)i;
}

__global__ void __launch_bounds__(256) count_keys_kernel(const int64_t* __restrict__ keys, int64_t E,
                                                         int64_t num_keys, int32_t* __restrict__ counts,
                                                         int32_t* __restrict__ err_flag) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= E) return;
  int64_t k = keys[i];
  if (k < 0 || k >= num_keys) {
    if (err_flag) atomicOr(err_flag, MT_FLAG_BAD_INDEX);
    return;
  }
  atomicAdd(&counts[k], 1);  // integer atomics: the result does not depend on the order
}

__global__ void __launch_bounds__(256) gather_i64_i32_kernel(const int64_t* __restrict__ src,
                                                             const int32_t* __restrict__ perm, int64_t n,
                                                             int32_t* __restrict__ out) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = (int32_t)src[perm ? perm[i] : i];
}

__global__ void __launch_bounds__(256) check_sorted_kernel(const int64_t* __restrict__ keys, int64_t n,
                                                           int32_t* __restrict__ err_flag) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i + 1 >= n) return;
  if (keys[i] > keys[i + 1]) atomicOr(err_flag, MT_FLAG_UNSORTED);
}

// =========================================================================
// a4: species embedding                 reference src/matten/nn/embedding.py:85-110
// =========================================================================
template <typename T>
__global__ void __launch_bounds__(256) species_embed_kernel(
    const int64_t* __restrict__ Z, int z_given, const int64_t* __restrict__ lut, int64_t min_z,
    int64_t max_z, int S, int dim, const T* __restrict__ lin_w, const T* __restrict__ lin_b, int64_t N,
    int64_t* __restrict__ species_index, T* __restrict__ attrs, T* __restrict__ feats,
    int32_t* __restrict__ err_flag) {
  // one warp per node
  int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (n >= N) return;
  int64_t s;
  if (z_given) {
    int64_t z = Z[n];
    s = (z < min_z || z > max_z) ? -1 : lut[z - min_z];
    if (s < 0) {
      if (err_flag && lane == 0) atomicOr(err_flag, MT_FLAG_BAD_SPECIES);
      s = 0;
    }
    if (species_index && lane == 0) species_index[n] = s;
  } else {
    s = species_index[n];
    if (s < 0 || s >= S) {
      if (err_flag && lane == 0) atomicOr(err_flag, MT_FLAG_BAD_SPECIES);
      s = 0;
    }
  }
  if (attrs)
    for (int j = lane; j < S; j += 32) attrs[n * S + j] = (j == s) ? T(1) : T(0);
  if (feats)
    for (int j = lane; j < dim; j += 32) feats[n * dim + j] = lin_w[(int64_t)j * S + s] + lin_b[j];
}


// =========================================================================
// periodic neighbour list (reference src/matten/data/data.py:285-413: ASE primitive_neighbor_list("ijS") with
// self_interaction=True, then the true self edges (i == j, S == 0) dropped).  All arithmetic in fp64, like the
// reference's numpy/ASE path.  Edges of centre i are emitted in the canonical order (j, Sx, Sy, Sz), centres in
// ascending order: the same order as matten_b200/data/neighbors.py.
// =========================================================================
struct NlGraph {
  double c[9];   // cell rows
  int R[3];      // images per axis: ceil(r_max / height) + span of the fractional coordinates
  int pad;
};

// The pair and the cell search derive the determinant, the fractional coordinates, the heights and the squared
// distance of a candidate (i, j, S) from these expressions alone, so that both compute the same bits for them.
__device__ __forceinline__ double nl_det(const double* c) {
  return c[0] * (c[4] * c[8] - c[5] * c[7]) - c[1] * (c[3] * c[8] - c[5] * c[6]) +
         c[2] * (c[3] * c[7] - c[4] * c[6]);
}

// inverse (adjugate / det): frac = pos @ inv(cell)
__device__ __forceinline__ void nl_inverse(const double* c, double det, double* inv) {
  inv[0] = (c[4] * c[8] - c[5] * c[7]) / det; inv[1] = (c[2] * c[7] - c[1] * c[8]) / det; inv[2] = (c[1] * c[5] - c[2] * c[4]) / det;
  inv[3] = (c[5] * c[6] - c[3] * c[8]) / det; inv[4] = (c[0] * c[8] - c[2] * c[6]) / det; inv[5] = (c[2] * c[3] - c[0] * c[5]) / det;
  inv[6] = (c[3] * c[7] - c[4] * c[6]) / det; inv[7] = (c[1] * c[6] - c[0] * c[7]) / det; inv[8] = (c[0] * c[4] - c[1] * c[3]) / det;
}

__device__ __forceinline__ double nl_frac(double x, double y, double z, const double* inv, int k) {
  return x * inv[k] + y * inv[3 + k] + z * inv[6 + k];
}

// distance between the lattice planes normal to axis k
__device__ __forceinline__ double nl_height(const double* c, double vol, int k) {
  const double* a = c + 3 * ((k + 1) % 3);
  const double* d = c + 3 * ((k + 2) % 3);
  const double cx = a[1] * d[2] - a[2] * d[1], cy = a[2] * d[0] - a[0] * d[2], cz = a[0] * d[1] - a[1] * d[0];
  return vol / sqrt(cx * cx + cy * cy + cz * cz);
}

// offset = S @ cell, then d = (pos[j] - pos[i]) + offset, |d|^2 = (dx^2 + dy^2) + dz^2 without contraction
__device__ __forceinline__ double nl_dist2(double dx0, double dy0, double dz0, int sx, int sy, int sz,
                                           const double* c) {
  const double ox = fma((double)sz, c[6], fma((double)sy, c[3], (double)sx * c[0]));
  const double oy = fma((double)sz, c[7], fma((double)sy, c[4], (double)sx * c[1]));
  const double oz = fma((double)sz, c[8], fma((double)sy, c[5], (double)sx * c[2]));
  const double dx = dx0 + ox, dy = dy0 + oy, dz = dz0 + oz;
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

template <typename T>
__global__ void __launch_bounds__(128) nl_setup_kernel(const T* __restrict__ pos, const T* __restrict__ cell,
                                                       const int64_t* __restrict__ ptr, int64_t B, double r_max,
                                                       NlGraph* __restrict__ out) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= B) return;
  NlGraph g;
  for (int k = 0; k < 9; ++k) g.c[k] = (double)cell[b * 9 + k];
  const double* c = g.c;
  const double det = nl_det(c);
  const double vol = fabs(det);
  int span = 0;
  if (vol > 0) {
    double inv[9];
    nl_inverse(c, det, inv);
    double fmin = 1e300, fmax = -1e300;
    for (int64_t i = ptr[b]; i < ptr[b + 1]; ++i) {
      const double x = (double)pos[i * 3], y = (double)pos[i * 3 + 1], z = (double)pos[i * 3 + 2];
      for (int k = 0; k < 3; ++k) {
        const double f = nl_frac(x, y, z, inv, k);
        fmin = f < fmin ? f : fmin;
        fmax = f > fmax ? f : fmax;
      }
    }
    if (ptr[b + 1] > ptr[b]) span = (int)ceil(fmax - fmin);
  }
  for (int k = 0; k < 3; ++k) g.R[k] = vol > 0 ? (int)ceil(r_max / nl_height(c, vol, k)) + span : 0;
  g.pad = 0;
  out[b] = g;
}

// FILL == false: counts[i] = number of neighbours of centre i; FILL == true: write them at offsets[i]
template <typename T, bool FILL>
__global__ void __launch_bounds__(128) nl_pairs_kernel(const T* __restrict__ pos, const int64_t* __restrict__ batch,
                                                       const int64_t* __restrict__ ptr,
                                                       const NlGraph* __restrict__ graphs, int64_t N, double r2,
                                                       int32_t* __restrict__ counts,
                                                       const int32_t* __restrict__ offsets,
                                                       int64_t* __restrict__ ei, int64_t E, T* __restrict__ shifts,
                                                       T* __restrict__ num_neigh) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int64_t b = batch ? batch[i] : 0;
  const NlGraph g = graphs[b];
  const double xi = (double)pos[i * 3], yi = (double)pos[i * 3 + 1], zi = (double)pos[i * 3 + 2];
  int64_t w = FILL ? offsets[i] : 0;
  int cnt = 0;
  for (int64_t j = ptr[b]; j < ptr[b + 1]; ++j) {
    const double dx0 = (double)pos[j * 3] - xi, dy0 = (double)pos[j * 3 + 1] - yi, dz0 = (double)pos[j * 3 + 2] - zi;
    for (int sx = -g.R[0]; sx <= g.R[0]; ++sx)
      for (int sy = -g.R[1]; sy <= g.R[1]; ++sy)
        for (int sz = -g.R[2]; sz <= g.R[2]; ++sz) {
          const double d2 = nl_dist2(dx0, dy0, dz0, sx, sy, sz, g.c);
          if (d2 < r2 && !(j == i && sx == 0 && sy == 0 && sz == 0)) {
            if (FILL) {
              ei[w] = i;
              ei[E + w] = j;
              shifts[w * 3] = (T)sx; shifts[w * 3 + 1] = (T)sy; shifts[w * 3 + 2] = (T)sz;
              ++w;
            }
            ++cnt;
          }
        }
  }
  if (FILL) { if (num_neigh) num_neigh[i] = (T)cnt; }
  else counts[i] = cnt;
}

// =========================================================================
// cell-list neighbour search: the same (i, j, S) set, order and outputs as nl_pairs_kernel, in time linear in the
// atoms of a crystal.  Binning is only a prefilter: a candidate (i, j, S) is accepted by nl_pairs_kernel's own
// expressions (nl_dist2 against r_max^2 in the original frame, the image bound |S_k| <= R_k with the same R_k).
//
// Periodic crystal (|det cell| > 0): fractional coordinates f are wrapped, n = floor(f), w = f - n, bin
// min(floor(w nb_k), nb_k - 1).  Bins are no thinner than r_max (1 + 2 eps) in each height h_k and the search covers
// D_k = ceil(r_max (1 + eps) nb_k / h_k) bins on each side, so every pair closer than r_max is found also when the
// cell is thinner than r_max (then nb_k = 1 and the window holds many images).  A window bin g maps to the wrapped
// bin g mod nb and the image T = floor(g / nb) of the wrapped frame; S = T - n_j + n_i in the original frame.
// Zero cell (no images): bins over the Cartesian bounding box of the crystal, D = 1, no wrapping.
// =========================================================================
constexpr double kNlEps = 1e-6;

struct NlCells {
  double c[9];         // cell rows
  double inv[9];       // inverse of the cell (periodic crystals)
  double lo[3];        // zero cell: lower corner of the bounding box
  double scale[3];     // bins per unit of the binning coordinate (periodic: nb; zero cell: nb / extent)
  uint64_t wprod;      // bins in the search window of a centre: (2 D0 + 1)(2 D1 + 1)(2 D2 + 1)
  int R[3];            // image bound of nl_pairs_kernel
  int nb[3];           // bins per axis
  int D[3];            // window half-width in bins
  int periodic;
};

// per atom: integer part of the fractional coordinates, and its bin in its crystal (-1: a non-finite coordinate)
struct NlCentre {
  int n[3];
  int bin;
};

// per bin-sorted atom: what a candidate test reads
struct NlAtom {
  double p[3];
  int j;
  int n[3];
};

// order-preserving map of a (non-NaN) double onto uint64, for atomicMin / atomicMax
__device__ __forceinline__ unsigned long long nl_ord(double v) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double nl_unord(unsigned long long u) {
  return __longlong_as_double((long long)((u >> 63) ? (u & 0x7fffffffffffffffull) : ~u));
}

__device__ __forceinline__ int nl_floor_div(int a, int n) { return a >= 0 ? a / n : -((-a + n - 1) / n); }

// binning coordinates of an atom: fractional (periodic crystal) or Cartesian (zero cell)
__device__ __forceinline__ void nl_cells_coords(const NlCells& g, double x, double y, double z, double* f) {
  if (g.periodic) {
#pragma unroll
    for (int k = 0; k < 3; ++k) f[k] = nl_frac(x, y, z, g.inv, k);
  } else {
    f[0] = x; f[1] = y; f[2] = z;
  }
}

// ext [B,6]: per axis min (0..2) and max (3..5) of the binning coordinates, starting at nl_setup_kernel's 1e300 / -1e300
template <typename T>
__global__ void __launch_bounds__(128) nl_cells_setup_kernel(const T* __restrict__ cell, int64_t B,
                                                             NlCells* __restrict__ cs,
                                                             unsigned long long* __restrict__ ext) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= B) return;
  NlCells g;
  for (int k = 0; k < 9; ++k) g.c[k] = (double)cell[b * 9 + k];
  const double det = nl_det(g.c);
  g.periodic = fabs(det) > 0;
  if (g.periodic) nl_inverse(g.c, det, g.inv);
  else
    for (int k = 0; k < 9; ++k) g.inv[k] = 0.0;
  cs[b] = g;
  for (int k = 0; k < 3; ++k) {
    ext[b * 6 + k] = nl_ord(1e300);
    ext[b * 6 + 3 + k] = nl_ord(-1e300);
  }
}

// min / max of the binning coordinates per crystal, NaN skipped (as nl_setup_kernel's comparisons skip it): a block
// of one crystal reduces in shared memory first, a block across crystals falls back to one atomic per atom and value
template <typename T>
__global__ void __launch_bounds__(256) nl_cells_extent_kernel(const T* __restrict__ pos,
                                                              const int64_t* __restrict__ batch, int64_t N,
                                                              const NlCells* __restrict__ cs,
                                                              unsigned long long* __restrict__ ext) {
  __shared__ double red[8][6];
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const bool valid = i < N;
  const int64_t b = valid && batch ? batch[i] : 0;
  double v[6] = {1e300, 1e300, 1e300, -1e300, -1e300, -1e300};
  if (valid) {
    double f[3];
    nl_cells_coords(cs[b], (double)pos[i * 3], (double)pos[i * 3 + 1], (double)pos[i * 3 + 2], f);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      v[k] = f[k] < v[k] ? f[k] : v[k];
      v[3 + k] = f[k] > v[3 + k] ? f[k] : v[3 + k];
    }
  }
  const int64_t b0 = batch ? batch[blockIdx.x * (int64_t)blockDim.x] : 0;
  if (__syncthreads_and(!valid || b == b0)) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      for (int o = 16; o > 0; o >>= 1) {
        const double u = __shfl_xor_sync(0xffffffffu, v[k], o);
        v[k] = k < 3 ? (u < v[k] ? u : v[k]) : (u > v[k] ? u : v[k]);
      }
      if (lane == 0) red[warp][k] = v[k];
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      const int k = threadIdx.x;
      double r = red[0][k];
      for (int w = 1; w < 8; ++w) r = k < 3 ? (red[w][k] < r ? red[w][k] : r) : (red[w][k] > r ? red[w][k] : r);
      if (k < 3) atomicMin(&ext[b0 * 6 + k], nl_ord(r));
      else atomicMax(&ext[b0 * 6 + k], nl_ord(r));
    }
  } else if (valid) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      atomicMin(&ext[b * 6 + k], nl_ord(v[k]));
      atomicMax(&ext[b * 6 + 3 + k], nl_ord(v[3 + k]));
    }
  }
}

// per crystal: nl_setup_kernel's R_k, then the bins (at most max(1, atoms) per crystal) and the search window.
// nbins[b] = bins of crystal b (scanned into bin offsets next); status != 0 if a window cannot be indexed in 64 bits.
__global__ void __launch_bounds__(128) nl_cells_grid_kernel(const int64_t* __restrict__ ptr, int64_t B, double r_max,
                                                            NlCells* __restrict__ cs,
                                                            const unsigned long long* __restrict__ ext,
                                                            int32_t* __restrict__ nbins, int32_t* __restrict__ status) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b == 0) nbins[B] = 0;
  if (b >= B) return;
  NlCells g = cs[b];
  const int64_t n = ptr[b + 1] - ptr[b];
  double lo[3], hi[3], len[3];
  for (int k = 0; k < 3; ++k) {
    lo[k] = nl_unord(ext[b * 6 + k]);
    hi[k] = nl_unord(ext[b * 6 + 3 + k]);
  }
  if (g.periodic) {
    const double f_lo = fmin(fmin(lo[0], lo[1]), lo[2]), f_hi = fmax(fmax(hi[0], hi[1]), hi[2]);
    const int span = n > 0 ? (int)ceil(f_hi - f_lo) : 0;
    const double vol = fabs(nl_det(g.c));
    for (int k = 0; k < 3; ++k) {
      len[k] = nl_height(g.c, vol, k);
      g.R[k] = (int)ceil(r_max / len[k]) + span;
    }
  } else {
    for (int k = 0; k < 3; ++k) {
      len[k] = hi[k] - lo[k];
      g.lo[k] = lo[k];
      g.R[k] = 0;
    }
  }
  const double cap = n > 1 ? (double)n : 1.0;
  double nb[3];
  for (int k = 0; k < 3; ++k) nb[k] = fmin(cap, fmax(1.0, floor(len[k] / (r_max * (1.0 + 2.0 * kNlEps)))));
  for (double prod = nb[0] * nb[1] * nb[2]; prod > cap; prod = nb[0] * nb[1] * nb[2]) {
    const int k = nb[0] >= nb[1] ? (nb[0] >= nb[2] ? 0 : 2) : (nb[1] >= nb[2] ? 1 : 2);
    nb[k] = fmax(1.0, fmin(nb[k] - 1.0, floor(nb[k] * cap / prod)));
  }
  double wprod = 1.0;
  bool ok = true;
  for (int k = 0; k < 3; ++k) {
    g.nb[k] = (int)nb[k];
    const double d = g.periodic ? ceil(r_max * (1.0 + kNlEps) * nb[k] / len[k]) : 1.0;
    ok = ok && d < 1e6;
    g.D[k] = ok ? (int)d : 1;
    g.scale[k] = g.periodic ? nb[k] : (len[k] > 0 ? nb[k] / len[k] : 0.0);
    wprod *= 2.0 * g.D[k] + 1.0;
  }
  // a fill entry packs (j - ptr[b]) * wprod + (window index) into 63 bits
  if (!ok || wprod * cap >= 4e18) atomicOr(status, 1);
  g.wprod = (uint64_t)wprod;
  cs[b] = g;
  nbins[b] = g.nb[0] * g.nb[1] * g.nb[2];
}

// keys[i] = global bin of atom i (bin0[b] + local bin), `sentinel` for an atom with a non-finite coordinate
template <typename T>
__global__ void __launch_bounds__(256) nl_cells_bin_kernel(const T* __restrict__ pos, const int64_t* __restrict__ batch,
                                                           int64_t N, const NlCells* __restrict__ cs,
                                                           const int32_t* __restrict__ bin0, int64_t sentinel,
                                                           int64_t* __restrict__ keys, NlCentre* __restrict__ cen) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= N) return;
  const int64_t b = batch ? batch[i] : 0;
  const NlCells& g = cs[b];
  double f[3];
  nl_cells_coords(g, (double)pos[i * 3], (double)pos[i * 3 + 1], (double)pos[i * 3 + 2], f);
  NlCentre a = {{0, 0, 0}, -1};
  int64_t key = sentinel;
  if (isfinite(f[0]) && isfinite(f[1]) && isfinite(f[2])) {
    int cb[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double w = f[k] - g.lo[k];
      if (g.periodic) {
        const double fl = floor(f[k]);
        a.n[k] = (int)fl;
        w = f[k] - fl;
      }
      const int c = (int)floor(w * g.scale[k]);
      cb[k] = c < 0 ? 0 : (c < g.nb[k] ? c : g.nb[k] - 1);
    }
    a.bin = (cb[0] * g.nb[1] + cb[1]) * g.nb[2] + cb[2];
    key = bin0[b] + a.bin;
  }
  keys[i] = key;
  cen[i] = a;
}

template <typename T>
__global__ void __launch_bounds__(256) nl_cells_gather_kernel(const T* __restrict__ pos, const int32_t* __restrict__ perm,
                                                              const NlCentre* __restrict__ cen, int64_t N,
                                                              NlAtom* __restrict__ rec) {
  const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (s >= N) return;
  const int j = perm[s];
  const NlCentre a = cen[j];
  rec[s] = {{(double)pos[(int64_t)j * 3], (double)pos[(int64_t)j * 3 + 1], (double)pos[(int64_t)j * 3 + 2]},
            j, {a.n[0], a.n[1], a.n[2]}};
}

// One thread per centre, centres in bin order (neighbouring threads search the same bins).  FILL == false: counts[i]
// = neighbours of centre i; FILL == true: entries (j - ptr[b]) * wprod + (window index) at offsets[i] in edge_index
// row 0, ordered by nl_cells_order_kernel, and num_neigh.
template <typename T, bool FILL>
__global__ void __launch_bounds__(128) nl_cells_pairs_kernel(
    const int64_t* __restrict__ batch, const int64_t* __restrict__ ptr, const NlCells* __restrict__ cs,
    const int32_t* __restrict__ bin0, const int32_t* __restrict__ rowptr, const NlAtom* __restrict__ rec,
    const NlCentre* __restrict__ cen, int64_t N, double r2, int32_t* __restrict__ counts,
    const int32_t* __restrict__ offsets, uint64_t* __restrict__ entries, T* __restrict__ num_neigh) {
  const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (s >= N) return;
  const NlAtom a = rec[s];
  const int i = a.j;
  const NlCentre ci = cen[i];
  int cnt = 0;
  if (ci.bin >= 0) {
    const int64_t b = batch ? batch[i] : 0;
    const NlCells& g = cs[b];
    double c[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) c[k] = g.c[k];
    const int nb0 = g.nb[0], nb1 = g.nb[1], nb2 = g.nb[2];
    const int D0 = g.D[0], D1 = g.D[1], D2 = g.D[2];
    const int R0 = g.R[0], R1 = g.R[1], R2 = g.R[2];
    const bool periodic = g.periodic;
    const uint64_t wprod = g.wprod;
    const int cz = ci.bin % nb2, cy = (ci.bin / nb2) % nb1, cx = ci.bin / (nb2 * nb1);
    const int64_t j0 = ptr[b];
    const int32_t* bp = rowptr + bin0[b];
    int64_t w = FILL ? offsets[i] : 0;
    uint64_t t = 0;  // window index, lexicographic in (gx, gy, gz)
    for (int gx = cx - D0; gx <= cx + D0; ++gx) {
      const int tx = periodic ? nl_floor_div(gx, nb0) : 0, bx = gx - tx * nb0;
      for (int gy = cy - D1; gy <= cy + D1; ++gy) {
        const int ty = periodic ? nl_floor_div(gy, nb1) : 0, by = gy - ty * nb1;
        for (int gz = cz - D2; gz <= cz + D2; ++gz, ++t) {
          const int tz = periodic ? nl_floor_div(gz, nb2) : 0, bz = gz - tz * nb2;
          if (bx < 0 || bx >= nb0 || by < 0 || by >= nb1 || bz < 0 || bz >= nb2) continue;  // zero cell only
          const int bin = (bx * nb1 + by) * nb2 + bz;
          for (int q = bp[bin], qe = bp[bin + 1]; q < qe; ++q) {
            const NlAtom o = rec[q];
            const int sx = tx - o.n[0] + ci.n[0], sy = ty - o.n[1] + ci.n[1], sz = tz - o.n[2] + ci.n[2];
            if (abs(sx) > R0 || abs(sy) > R1 || abs(sz) > R2) continue;
            const double d2 = nl_dist2(o.p[0] - a.p[0], o.p[1] - a.p[1], o.p[2] - a.p[2], sx, sy, sz, c);
            if (d2 < r2 && !(o.j == i && sx == 0 && sy == 0 && sz == 0)) {
              if (FILL) entries[w++] = (uint64_t)(o.j - j0) * wprod + t;
              ++cnt;
            }
          }
        }
      }
    }
  }
  if (FILL) { if (num_neigh) num_neigh[i] = (T)cnt; }
  else counts[i] = cnt;
}

// One warp per centre: the rank of every entry among the centre's entries (all distinct) is its place in the
// canonical (j, Sx, Sy, Sz) order -- the window index is lexicographic in the wrapped image T, and S = T - n_j + n_i.
// Writes edge_index row 1 and the shifts at that place, then overwrites the entries with the centre.  Any degree.
template <typename T>
__global__ void __launch_bounds__(256) nl_cells_order_kernel(const int64_t* __restrict__ batch,
                                                             const int64_t* __restrict__ ptr,
                                                             const NlCells* __restrict__ cs,
                                                             const NlCentre* __restrict__ cen,
                                                             const int32_t* __restrict__ offsets, int64_t N, int64_t E,
                                                             int64_t* __restrict__ ei, T* __restrict__ shifts) {
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= N) return;
  const int64_t beg = offsets[i], end = offsets[i + 1];
  if (beg == end) return;
  const int64_t b = batch ? batch[i] : 0;
  const NlCells& g = cs[b];
  const NlCentre ci = cen[i];
  const int nb0 = g.nb[0], nb1 = g.nb[1], nb2 = g.nb[2];
  const int W1 = 2 * g.D[1] + 1, W2 = 2 * g.D[2] + 1;
  const uint64_t wprod = g.wprod;
  const int cz = ci.bin % nb2, cy = (ci.bin / nb2) % nb1, cx = ci.bin / (nb2 * nb1);
  const int64_t j0 = ptr[b];
  const uint64_t* entries = reinterpret_cast<const uint64_t*>(ei);
  for (int64_t p0 = beg; p0 < end; p0 += 32) {
    const int64_t p = p0 + lane;
    const uint64_t key = p < end ? entries[p] : ~0ull;
    int64_t rank = 0;
    for (int64_t q0 = beg; q0 < end; q0 += 32) {
      const uint64_t kq = q0 + lane < end ? entries[q0 + lane] : ~0ull;
#pragma unroll 8
      for (int l = 0; l < 32; ++l) rank += __shfl_sync(0xffffffffu, kq, l) < key;
    }
    if (p < end) {
      const int64_t j = j0 + (int64_t)(key / wprod);
      uint64_t t = key % wprod;
      const int tz = (int)(t % W2);
      t /= W2;
      const int ty = (int)(t % W1), tx = (int)(t / W1);
      const int gx = cx - g.D[0] + tx, gy = cy - g.D[1] + ty, gz = cz - g.D[2] + tz;
      const NlCentre cj = cen[j];
      int S[3] = {0, 0, 0};
      if (g.periodic) {
        S[0] = nl_floor_div(gx, nb0) - cj.n[0] + ci.n[0];
        S[1] = nl_floor_div(gy, nb1) - cj.n[1] + ci.n[1];
        S[2] = nl_floor_div(gz, nb2) - cj.n[2] + ci.n[2];
      }
      const int64_t e = beg + rank;
      ei[E + e] = j;
#pragma unroll
      for (int k = 0; k < 3; ++k) shifts[e * 3 + k] = (T)S[k];
    }
  }
  __syncwarp();
  for (int64_t p = beg + lane; p < end; p += 32) ei[p] = i;
}

// offsets[N] = -1 when the int32 scan of the counts wrapped (2^31 edges or more) or a window could not be indexed
__global__ void __launch_bounds__(256) nl_cells_total_kernel(int32_t* __restrict__ offsets, int64_t N,
                                                             const int32_t* __restrict__ status) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= N) return;
  if (offsets[i + 1] < offsets[i] || *status != 0) offsets[N] = -1;
}

}  // namespace mt

// ===========================================================================
// C ABI
// ===========================================================================
using namespace mt;

static inline unsigned grid_for(int64_t n, int threads) { return (unsigned)ceil_div<int64_t>(n, threads); }
static int csr_by_key_run(const int64_t* keys, int64_t E, int64_t num_keys, int32_t* rowptr, int32_t* perm,
                          void* workspace, int32_t* err_flag, cudaStream_t st);

extern "C" {

int mt_edge_vectors(int dtype, const void* pos, const int64_t* edge_index, const void* edge_cell_shift,
                    const void* cell, const int64_t* batch, int64_t N, int64_t E, int64_t B,
                    void* edge_vec, void* edge_len, int32_t* err_flag, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(N >= 0 && E >= 0 && B >= 0, "negative size");
  MT_REQUIRE((cell == nullptr) == (edge_cell_shift == nullptr), "cell and edge_cell_shift must be given together");
  MT_REQUIRE(!(cell != nullptr && B > 1 && batch == nullptr), "batch is required when the cell has a batch dimension");
  if (E == 0) return MT_OK;
  MT_REQUIRE(pos && edge_index, "null input");
  MT_DISPATCH_DTYPE(dtype, {
    edge_vectors_kernel<T><<<grid_for(E, 256), 256, 0, as_stream(stream)>>>(
        (const T*)pos, edge_index, (const T*)edge_cell_shift, (const T*)cell, batch, N, E, B, (T*)edge_vec,
        (T*)edge_len, err_flag);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_edge_sh(int dtype, const void* edge_vec, int64_t E, int lmax, int normalize, void* edge_sh,
               mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(lmax >= 0 && lmax <= MT_LMAX, "lmax %d not supported (0..%d)", lmax, MT_LMAX);
  if (E == 0) return MT_OK;
  MT_REQUIRE(edge_vec && edge_sh, "null pointer");
  cudaStream_t st = as_stream(stream);
  unsigned g = grid_for(E, 256);
#define MT_SH_CASE(L)                                                                          \
  case L:                                                                                      \
    edge_sh_kernel<T, L><<<g, 256, 0, st>>>((const T*)edge_vec, E, normalize, (T*)edge_sh);    \
    break;
  MT_DISPATCH_DTYPE(dtype, {
    switch (lmax) {
      MT_SH_CASE(0) MT_SH_CASE(1) MT_SH_CASE(2) MT_SH_CASE(3) MT_SH_CASE(4)
    }
  });
#undef MT_SH_CASE
  MT_LAUNCH_OK();
  return MT_OK;
}

// Without cutoff the centres of modes 3-5 are linspace(start, end, n), and their spacing needs n >= 2.
static inline bool centred_basis_ok(int mode, int num_basis, int cutoff) {
  return cutoff || num_basis >= 2 || mode < 3 || mode > 5;
}

int mt_edge_radial(int dtype, const void* edge_len, int64_t E, int mode, int num_basis, double start,
                   double end, int cutoff, double poly_p, const void* bessel_w, void* edge_emb,
                   mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(mode >= 0 && mode <= 6, "radial mode %d", mode);
  MT_REQUIRE(num_basis > 0 && end > start, "bad radial basis parameters");
  MT_REQUIRE(centred_basis_ok(mode, num_basis, cutoff), "radial mode %d without cutoff needs num_basis >= 2", mode);
  if (E == 0) return MT_OK;
  MT_REQUIRE(edge_len && edge_emb, "null pointer");
  MT_DISPATCH_DTYPE(dtype, {
    edge_radial_kernel<T><<<grid_for(E * num_basis, 256), 256, 0, as_stream(stream)>>>(
        (const T*)edge_len, E, mode, num_basis, (T)start, (T)end, cutoff, (T)poly_p, (const T*)bessel_w,
        (T*)edge_emb);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_edge_sh_bwd(int dtype, const void* edge_vec, const void* grad_sh, int64_t E, int lmax, int normalize,
                   void* grad_vec, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(lmax >= 0 && lmax <= MT_LMAX, "lmax %d not supported (0..%d)", lmax, MT_LMAX);
  MT_REQUIRE(E >= 0, "negative size");
  if (E == 0) return MT_OK;
  MT_REQUIRE(edge_vec && grad_sh && grad_vec, "null pointer");
  cudaStream_t st = as_stream(stream);
  unsigned g = grid_for(E, 256);
#define MT_SH_BWD_CASE(L)                                                                                       \
  case L:                                                                                                       \
    edge_sh_bwd_kernel<T, L><<<g, 256, 0, st>>>((const T*)edge_vec, (const T*)grad_sh, E, normalize, (T*)grad_vec); \
    break;
  MT_DISPATCH_DTYPE(dtype, {
    switch (lmax) {
      MT_SH_BWD_CASE(0) MT_SH_BWD_CASE(1) MT_SH_BWD_CASE(2) MT_SH_BWD_CASE(3) MT_SH_BWD_CASE(4)
    }
  });
#undef MT_SH_BWD_CASE
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_edge_radial_bwd(int dtype, const void* edge_len, const void* grad_emb, int64_t E, int mode, int num_basis,
                       double start, double end, int cutoff, double poly_p, const void* bessel_w, void* grad_len,
                       mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(mode == 0 || mode == 1 || (mode >= 3 && mode <= 6), "radial backward mode %d", mode);
  MT_REQUIRE(num_basis > 0 && end > start && E >= 0, "bad radial basis parameters");
  MT_REQUIRE(centred_basis_ok(mode, num_basis, cutoff), "radial mode %d without cutoff needs num_basis >= 2", mode);
  if (E == 0) return MT_OK;
  MT_REQUIRE(edge_len && grad_emb && grad_len, "null pointer");
  MT_DISPATCH_DTYPE(dtype, {
    edge_radial_bwd_kernel<T><<<grid_for(E, 256), 256, 0, as_stream(stream)>>>(
        (const T*)edge_len, (const T*)grad_emb, E, mode, num_basis, (T)start, (T)end, cutoff, (T)poly_p,
        (const T*)bessel_w, (T*)grad_len);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

size_t mt_edge_vectors_bwd_workspace_bytes(int dtype, int64_t E, int64_t B) {
  const size_t es = dtype == MT_F64 ? 8 : 4;
  if (E < 0) E = 0;
  if (B < 1) B = 1;
  return align256((size_t)E * 3 * es) + align256((size_t)E * 9 * es) + align256((size_t)(B + 1) * 4);
}

int mt_edge_vectors_bwd(int dtype, const void* edge_vec, const void* grad_vec, const void* grad_len,
                        const void* edge_cell_shift, const int32_t* rowptr, const int32_t* perm,
                        const int32_t* sender_ptr, const int32_t* sender_perm, const int32_t* graph_ptr, int64_t N,
                        int64_t E, int64_t B, void* grad_pos, void* grad_cell, void* workspace,
                        size_t workspace_bytes, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(N >= 0 && E >= 0 && B >= 0, "negative size");
  MT_REQUIRE(grad_cell == nullptr || edge_cell_shift != nullptr, "grad_cell needs edge_cell_shift");
  MT_REQUIRE(grad_cell == nullptr || B == 1 || graph_ptr != nullptr, "graph_ptr is required for more than one graph");
  cudaStream_t st = as_stream(stream);
  const size_t es = dtype == MT_F64 ? 8 : 4;
  if (E == 0) {
    if (grad_pos) MT_CUDA_OK(cudaMemsetAsync(grad_pos, 0, (size_t)N * 3 * es, st));
    if (grad_cell) MT_CUDA_OK(cudaMemsetAsync(grad_cell, 0, (size_t)B * 9 * es, st));
    return MT_OK;
  }
  if (grad_pos == nullptr && grad_cell == nullptr) return MT_OK;
  MT_REQUIRE(edge_vec && rowptr && perm && sender_ptr && sender_perm, "null pointer");
  MT_REQUIRE(workspace != nullptr && workspace_bytes >= mt_edge_vectors_bwd_workspace_bytes(dtype, E, B),
             "edge_vectors_bwd workspace too small");
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  void* dvs = ws;
  void* sdv = grad_cell ? ws + align256((size_t)E * 3 * es) : nullptr;
  int32_t* cptr = reinterpret_cast<int32_t*>(ws + align256((size_t)E * 3 * es) + align256((size_t)E * 9 * es));
  MT_DISPATCH_DTYPE(dtype, {
    edge_dv_kernel<T><<<grid_for(E, 256), 256, 0, st>>>((const T*)edge_vec, (const T*)grad_vec, (const T*)grad_len,
                                                        (const T*)edge_cell_shift, perm, E, (T*)dvs, (T*)sdv);
  });
  MT_LAUNCH_OK();
  if (grad_pos && N > 0) {
    MT_DISPATCH_DTYPE(dtype, {
      pos_grad_kernel<T><<<grid_for(N, 256), 256, 0, st>>>((const T*)dvs, rowptr, sender_ptr, sender_perm, N,
                                                           (T*)grad_pos);
    });
    MT_LAUNCH_OK();
  }
  if (grad_cell && B > 0) {
    graph_edge_ptr_kernel<<<grid_for(B + 1, 256), 256, 0, st>>>(sender_ptr, graph_ptr, B, N, cptr);
    MT_LAUNCH_OK();
    return mt_segment_sum_gather(dtype, sdv, sender_perm, cptr, 9, B, E, grad_cell, stream);
  }
  return MT_OK;
}

size_t mt_csr_workspace_bytes(int64_t num_keys, int64_t E) {
  if (E < 0) E = 0;
  if (num_keys < 0) num_keys = 0;
  int64_t nblocks = ceil_div<int64_t>(E > 0 ? E : 1, kSortTile);
  size_t hist = (size_t)256 * nblocks;
  size_t scan_n = hist > (size_t)(num_keys + 1) ? hist : (size_t)(num_keys + 1);
  size_t b = 0;
  b += 4 * align256((size_t)E * 4);                    // k0 k1 v0 v1
  b += align256(hist * 4);                             // histogram
  b += align256(scan_tmp_elems((int64_t)scan_n) * 4);  // scan temporaries
  return b + 256;
}

int mt_csr_by_key(const int64_t* keys, int64_t E, int64_t num_keys, int32_t* rowptr, int32_t* perm,
                  void* workspace, size_t workspace_bytes, int32_t* err_flag, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(E >= 0 && num_keys >= 0 && rowptr, "bad arguments");
  MT_REQUIRE(E < (int64_t)2147483647 && num_keys < (int64_t)2147483647, "sizes must fit int32");
  MT_REQUIRE(workspace_bytes >= mt_csr_workspace_bytes(num_keys, E), "workspace too small");
  cudaStream_t st = as_stream(stream);
  if (E == 0) {
    MT_CUDA_OK(cudaMemsetAsync(rowptr, 0, (size_t)(num_keys + 1) * 4, st));
    return MT_OK;
  }
  MT_REQUIRE(keys && workspace, "null pointer");
  return csr_by_key_run(keys, E, num_keys, rowptr, perm, workspace, err_flag, st);
}

}  // extern "C"

// the stable radix sort behind mt_csr_by_key (checked arguments, E > 0)
static int csr_by_key_run(const int64_t* keys, int64_t E, int64_t num_keys, int32_t* rowptr, int32_t* perm,
                          void* workspace, int32_t* err_flag, cudaStream_t st) {
  char* ws = (char*)workspace;
  size_t eb = align256((size_t)E * 4);
  int32_t* k0 = (int32_t*)ws;
  int32_t* k1 = (int32_t*)(ws + eb);
  int32_t* v0 = (int32_t*)(ws + 2 * eb);
  int32_t* v1 = (int32_t*)(ws + 3 * eb);
  int nblocks = (int)ceil_div<int64_t>(E, kSortTile);
  size_t hist_n = (size_t)256 * nblocks;
  int32_t* hist = (int32_t*)(ws + 4 * eb);
  int32_t* stmp = (int32_t*)(ws + 4 * eb + align256(hist_n * 4));

  if (perm == nullptr) {
    // row pointers only: histogram + scan
    MT_CUDA_OK(cudaMemsetAsync(rowptr, 0, (size_t)(num_keys + 1) * 4, st));
    count_keys_kernel<<<grid_for(E, 256), 256, 0, st>>>(keys, E, num_keys, rowptr, err_flag);
    MT_LAUNCH_OK();
    return exclusive_scan_i32(rowptr, num_keys + 1, stmp, st);
  }

  keys_init_kernel<<<grid_for(E, 256), 256, 0, st>>>(keys, E, num_keys, k0, v0, err_flag);
  MT_LAUNCH_OK();
  int bits = 1;
  while (((int64_t)1 << bits) < num_keys) ++bits;
  int passes = (bits + 7) / 8;
  int32_t *ki = k0, *vi = v0, *ko = k1, *vo = v1;
  for (int p = 0; p < passes; ++p) {
    bool last = (p == passes - 1);
    radix_hist_kernel<<<nblocks, kSortThreads, 0, st>>>(ki, E, 8 * p, hist, nblocks);
    MT_LAUNCH_OK();
    int rc = exclusive_scan_i32(hist, (int64_t)hist_n, stmp, st);
    if (rc != MT_OK) return rc;
    radix_scatter_kernel<<<nblocks, kSortThreads, 0, st>>>(ki, vi, E, 8 * p, hist, nblocks, ko,
                                                           last ? perm : vo);
    MT_LAUNCH_OK();
    int32_t* t;
    t = ki; ki = ko; ko = t;
    t = vi; vi = vo; vo = t;
  }
  // ki now holds the sorted keys
  rowptr_from_sorted_kernel<<<grid_for(E + 1, 256), 256, 0, st>>>(ki, E, num_keys, rowptr);
  MT_LAUNCH_OK();
  return MT_OK;
}

extern "C" {

int mt_gather_i64_to_i32(const int64_t* src, const int32_t* perm, int64_t n, int32_t* out,
                         mt_stream stream) {
  MT_ENTRY_GUARD();
  if (n <= 0) return MT_OK;
  MT_REQUIRE(src && out, "null pointer");
  gather_i64_i32_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(src, perm, n, out);
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_check_sorted(const int64_t* keys, int64_t n, int32_t* err_flag, mt_stream stream) {
  MT_ENTRY_GUARD();
  if (n <= 1) return MT_OK;
  MT_REQUIRE(keys && err_flag, "null pointer");
  check_sorted_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(keys, n, err_flag);
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_species_embed(int dtype, const int64_t* atomic_numbers, int z_given, const int64_t* lut,
                     int64_t min_z, int64_t max_z, int num_species, int dim, const void* lin_w,
                     const void* lin_b, int64_t N, int64_t* species_index, void* node_attrs,
                     void* node_feats, int32_t* err_flag, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(num_species > 0 && dim >= 0, "bad sizes");
  if (N == 0) return MT_OK;
  if (z_given) MT_REQUIRE(atomic_numbers && lut, "atomic_numbers and lut required");
  else MT_REQUIRE(species_index, "species_index required when z_given == 0");
  if (node_feats) MT_REQUIRE(lin_w && lin_b, "linear weights required");
  MT_DISPATCH_DTYPE(dtype, {
    species_embed_kernel<T><<<grid_for(N * 32, 256), 256, 0, as_stream(stream)>>>(
        atomic_numbers, z_given, lut, min_z, max_z, num_species, dim, (const T*)lin_w, (const T*)lin_b, N,
        species_index, (T*)node_attrs, (T*)node_feats, err_flag);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}


size_t mt_neighbor_workspace_bytes(int64_t N, int64_t B) {
  return ((size_t)(B > 0 ? B : 1) * sizeof(NlGraph) + 255) / 256 * 256 + (scan_tmp_elems(N + 1) + 8) * sizeof(int32_t);
}

int mt_neighbor_count(int dtype, const void* pos, const void* cell, const int64_t* batch, const int64_t* ptr,
                      int64_t N, int64_t B, double r_max, int32_t* offsets, void* workspace, size_t workspace_bytes,
                      mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(N >= 0 && B >= 1 && r_max > 0, "bad arguments");
  MT_REQUIRE(pos && cell && ptr && offsets && workspace, "null pointer");
  MT_REQUIRE(B == 1 || batch != nullptr, "batch vector required for more than one graph");
  MT_REQUIRE(workspace_bytes >= mt_neighbor_workspace_bytes(N, B), "neighbour-list workspace too small");
  cudaStream_t st = as_stream(stream);
  NlGraph* graphs = static_cast<NlGraph*>(workspace);
  int32_t* tmp = reinterpret_cast<int32_t*>(static_cast<unsigned char*>(workspace) +
                                            ((size_t)B * sizeof(NlGraph) + 255) / 256 * 256);
  MT_DISPATCH_DTYPE(dtype, {
    nl_setup_kernel<T><<<grid_for(B, 128), 128, 0, st>>>((const T*)pos, (const T*)cell, ptr, B, r_max, graphs);
  });
  MT_LAUNCH_OK();
  MT_CUDA_OK(cudaMemsetAsync(offsets + N, 0, sizeof(int32_t), st));
  if (N > 0) {
    MT_DISPATCH_DTYPE(dtype, {
      nl_pairs_kernel<T, false><<<grid_for(N, 128), 128, 0, st>>>((const T*)pos, batch, ptr, graphs, N, r_max * r_max,
                                                                   offsets, nullptr, nullptr, 0, nullptr, nullptr);
    });
    MT_LAUNCH_OK();
  }
  return exclusive_scan_i32(offsets, N + 1, tmp, st);  // offsets[N] = number of edges
}

int mt_neighbor_fill(int dtype, const void* pos, const int64_t* batch, const int64_t* ptr, int64_t N, int64_t B,
                     double r_max, const int32_t* offsets, const void* workspace, int64_t* edge_index,
                     void* edge_cell_shift, void* num_neigh, int64_t E, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(N >= 0 && B >= 1 && E >= 0, "bad arguments");
  if (N == 0) return MT_OK;
  MT_REQUIRE(pos && ptr && offsets && workspace, "null pointer");
  MT_REQUIRE(E == 0 || (edge_index && edge_cell_shift), "null output pointer");
  const NlGraph* graphs = static_cast<const NlGraph*>(workspace);
  MT_DISPATCH_DTYPE(dtype, {
    nl_pairs_kernel<T, true><<<grid_for(N, 128), 128, 0, as_stream(stream)>>>(
        (const T*)pos, batch, ptr, graphs, N, r_max * r_max, nullptr, offsets, edge_index, E, (T*)edge_cell_shift,
        (T*)num_neigh);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}


// Workspace of the cell search, shared by count and fill; sized from N and B alone (at most N + B bins in all).
struct NlCellsLayout {
  size_t cells, ext, bin0, status, keys, rowptr, perm, cen, rec, scan, csr, total;
  NlCellsLayout(int64_t N, int64_t B) {
    if (N < 0) N = 0;
    if (B < 1) B = 1;
    size_t o = 0;
    auto take = [&o](size_t bytes) { const size_t at = o; o += align256(bytes); return at; };
    cells = take((size_t)B * sizeof(NlCells));
    ext = take((size_t)B * 6 * sizeof(unsigned long long));
    bin0 = take((size_t)(B + 1) * 4);
    status = take(4);
    keys = take((size_t)N * 8);
    rowptr = take((size_t)(N + B + 2) * 4);
    perm = take((size_t)N * 4);
    cen = take((size_t)N * sizeof(NlCentre));
    rec = take((size_t)N * sizeof(NlAtom));
    scan = take(scan_tmp_elems((N > B ? N : B) + 1) * 4);
    csr = take(mt_csr_workspace_bytes(N + B + 1, N));
    total = o;
  }
};

size_t mt_neighbor_cells_workspace_bytes(int64_t N, int64_t B) { return NlCellsLayout(N, B).total; }

int mt_neighbor_cells_count(int dtype, const void* pos, const void* cell, const int64_t* batch, const int64_t* ptr,
                            int64_t N, int64_t B, double r_max, int32_t* offsets, void* workspace,
                            size_t workspace_bytes, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(N >= 0 && B >= 1 && r_max > 0, "bad arguments");
  MT_REQUIRE(N + B + 2 < (int64_t)2147483647, "N + B must fit int32");
  MT_REQUIRE(pos && cell && ptr && offsets && workspace, "null pointer");
  MT_REQUIRE(B == 1 || batch != nullptr, "batch vector required for more than one graph");
  MT_REQUIRE(workspace_bytes >= mt_neighbor_cells_workspace_bytes(N, B), "neighbour-list workspace too small");
  cudaStream_t st = as_stream(stream);
  const NlCellsLayout L(N, B);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  NlCells* cs = reinterpret_cast<NlCells*>(ws + L.cells);
  unsigned long long* ext = reinterpret_cast<unsigned long long*>(ws + L.ext);
  int32_t* bin0 = reinterpret_cast<int32_t*>(ws + L.bin0);
  int32_t* status = reinterpret_cast<int32_t*>(ws + L.status);
  int64_t* keys = reinterpret_cast<int64_t*>(ws + L.keys);
  int32_t* rowptr = reinterpret_cast<int32_t*>(ws + L.rowptr);
  int32_t* perm = reinterpret_cast<int32_t*>(ws + L.perm);
  NlCentre* cen = reinterpret_cast<NlCentre*>(ws + L.cen);
  NlAtom* rec = reinterpret_cast<NlAtom*>(ws + L.rec);
  int32_t* tmp = reinterpret_cast<int32_t*>(ws + L.scan);
  MT_CUDA_OK(cudaMemsetAsync(offsets + N, 0, sizeof(int32_t), st));
  if (N == 0) return MT_OK;
  MT_CUDA_OK(cudaMemsetAsync(status, 0, sizeof(int32_t), st));
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_setup_kernel<T><<<grid_for(B, 128), 128, 0, st>>>((const T*)cell, B, cs, ext);
  });
  MT_LAUNCH_OK();
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_extent_kernel<T><<<grid_for(N, 256), 256, 0, st>>>((const T*)pos, batch, N, cs, ext);
  });
  MT_LAUNCH_OK();
  nl_cells_grid_kernel<<<grid_for(B, 128), 128, 0, st>>>(ptr, B, r_max, cs, ext, bin0, status);
  MT_LAUNCH_OK();
  int rc = exclusive_scan_i32(bin0, B + 1, tmp, st);
  if (rc != MT_OK) return rc;
  const int64_t sentinel = N + B;  // bins of all crystals number at most N + B
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_bin_kernel<T><<<grid_for(N, 256), 256, 0, st>>>((const T*)pos, batch, N, cs, bin0, sentinel, keys, cen);
  });
  MT_LAUNCH_OK();
  rc = csr_by_key_run(keys, N, sentinel + 1, rowptr, perm, ws + L.csr, nullptr, st);
  if (rc != MT_OK) return rc;
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_gather_kernel<T><<<grid_for(N, 256), 256, 0, st>>>((const T*)pos, perm, cen, N, rec);
  });
  MT_LAUNCH_OK();
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_pairs_kernel<T, false><<<grid_for(N, 128), 128, 0, st>>>(batch, ptr, cs, bin0, rowptr, rec, cen, N,
                                                                       r_max * r_max, offsets, nullptr, nullptr,
                                                                       nullptr);
  });
  MT_LAUNCH_OK();
  rc = exclusive_scan_i32(offsets, N + 1, tmp, st);  // offsets[N] = number of edges
  if (rc != MT_OK) return rc;
  nl_cells_total_kernel<<<grid_for(N, 256), 256, 0, st>>>(offsets, N, status);
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_neighbor_cells_fill(int dtype, const void* pos, const int64_t* batch, const int64_t* ptr, int64_t N, int64_t B,
                           double r_max, const int32_t* offsets, const void* workspace, int64_t* edge_index,
                           void* edge_cell_shift, void* num_neigh, int64_t E, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(N >= 0 && B >= 1, "bad arguments");
  MT_REQUIRE(E >= 0 && E < (int64_t)2147483647,
             "the cell search found 2^31 edges or more, or a cell too thin to search (offsets[N] = %lld)",
             (long long)E);
  if (N == 0) return MT_OK;
  MT_REQUIRE(pos && ptr && offsets && workspace, "null pointer");
  MT_REQUIRE(E == 0 || (edge_index && edge_cell_shift), "null output pointer");
  cudaStream_t st = as_stream(stream);
  const NlCellsLayout L(N, B);
  const unsigned char* ws = static_cast<const unsigned char*>(workspace);
  const NlCells* cs = reinterpret_cast<const NlCells*>(ws + L.cells);
  const int32_t* bin0 = reinterpret_cast<const int32_t*>(ws + L.bin0);
  const int32_t* rowptr = reinterpret_cast<const int32_t*>(ws + L.rowptr);
  const NlCentre* cen = reinterpret_cast<const NlCentre*>(ws + L.cen);
  const NlAtom* rec = reinterpret_cast<const NlAtom*>(ws + L.rec);
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_pairs_kernel<T, true><<<grid_for(N, 128), 128, 0, st>>>(
        batch, ptr, cs, bin0, rowptr, rec, cen, N, r_max * r_max, nullptr, offsets,
        reinterpret_cast<uint64_t*>(edge_index), (T*)num_neigh);
  });
  MT_LAUNCH_OK();
  if (E == 0) return MT_OK;
  MT_DISPATCH_DTYPE(dtype, {
    nl_cells_order_kernel<T><<<grid_for(N * 32, 256), 256, 0, st>>>(batch, ptr, cs, cen, offsets, N, E, edge_index,
                                                                     (T*)edge_cell_shift);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

}  // extern "C"
