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

template <typename T>
__global__ void __launch_bounds__(128) nl_setup_kernel(const T* __restrict__ pos, const T* __restrict__ cell,
                                                       const int64_t* __restrict__ ptr, int64_t B, double r_max,
                                                       NlGraph* __restrict__ out) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= B) return;
  NlGraph g;
  for (int k = 0; k < 9; ++k) g.c[k] = (double)cell[b * 9 + k];
  const double* c = g.c;
  const double det = c[0] * (c[4] * c[8] - c[5] * c[7]) - c[1] * (c[3] * c[8] - c[5] * c[6]) +
                     c[2] * (c[3] * c[7] - c[4] * c[6]);
  const double vol = fabs(det);
  int span = 0;
  if (vol > 0) {
    // inverse (adjugate / det): frac = pos @ inv(cell)
    double inv[9];
    inv[0] = (c[4] * c[8] - c[5] * c[7]) / det; inv[1] = (c[2] * c[7] - c[1] * c[8]) / det; inv[2] = (c[1] * c[5] - c[2] * c[4]) / det;
    inv[3] = (c[5] * c[6] - c[3] * c[8]) / det; inv[4] = (c[0] * c[8] - c[2] * c[6]) / det; inv[5] = (c[2] * c[3] - c[0] * c[5]) / det;
    inv[6] = (c[3] * c[7] - c[4] * c[6]) / det; inv[7] = (c[1] * c[6] - c[0] * c[7]) / det; inv[8] = (c[0] * c[4] - c[1] * c[3]) / det;
    double fmin = 1e300, fmax = -1e300;
    for (int64_t i = ptr[b]; i < ptr[b + 1]; ++i) {
      const double x = (double)pos[i * 3], y = (double)pos[i * 3 + 1], z = (double)pos[i * 3 + 2];
      for (int k = 0; k < 3; ++k) {
        const double f = x * inv[k] + y * inv[3 + k] + z * inv[6 + k];
        fmin = f < fmin ? f : fmin;
        fmax = f > fmax ? f : fmax;
      }
    }
    if (ptr[b + 1] > ptr[b]) span = (int)ceil(fmax - fmin);
  }
  for (int k = 0; k < 3; ++k) {
    int r = 0;
    if (vol > 0) {
      const double* a = c + 3 * ((k + 1) % 3);
      const double* d = c + 3 * ((k + 2) % 3);
      const double cx = a[1] * d[2] - a[2] * d[1], cy = a[2] * d[0] - a[0] * d[2], cz = a[0] * d[1] - a[1] * d[0];
      const double height = vol / sqrt(cx * cx + cy * cy + cz * cz);
      r = (int)ceil(r_max / height) + span;
    }
    g.R[k] = r;
  }
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
          // offset = S @ cell, then d = (pos[j] - pos[i]) + offset, |d|^2 = (dx^2 + dy^2) + dz^2 without contraction
          const double ox = fma((double)sz, g.c[6], fma((double)sy, g.c[3], (double)sx * g.c[0]));
          const double oy = fma((double)sz, g.c[7], fma((double)sy, g.c[4], (double)sx * g.c[1]));
          const double oz = fma((double)sz, g.c[8], fma((double)sy, g.c[5], (double)sx * g.c[2]));
          const double dx = dx0 + ox, dy = dy0 + oy, dz = dz0 + oz;
          const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
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

}  // namespace mt

// ===========================================================================
// C ABI
// ===========================================================================
using namespace mt;

static inline unsigned grid_for(int64_t n, int threads) { return (unsigned)ceil_div<int64_t>(n, threads); }

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

}  // extern "C"
