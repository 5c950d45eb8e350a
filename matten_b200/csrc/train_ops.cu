// Training-side kernels: backward of the node-side ops (species-indexed linear, Gate, pooling), training-mode
// BatchNorm reductions, loss and optimiser.  See include/matten_b200.h for the contract of every entry point.
// Everything here is deterministic: reductions are per-CTA partial sums combined in a fixed order.
#include "common.cuh"

namespace mt {

constexpr int kWgMaxBlocks = 64;
constexpr int kWgSplits = 16;   // node-range splits per (block, species) -> partial buffers (large weights)
constexpr int kWgSplitsSmall = 128;  // ... for weights of <= kWgSmallNumel elements (species-free linears: few CTAs otherwise)
constexpr int64_t kWgSmallNumel = 16384;
static inline int wg_max_splits(int64_t weight_numel) { return weight_numel <= kWgSmallNumel ? kWgSplitsSmall : kWgSplits; }
constexpr int kWgTile = 64;     // (u, w) tile
constexpr int kWgRows = 32;     // (node, m) rows staged per step

struct WgParams {
  int num_blocks;
  int32_t in_off[kWgMaxBlocks], out_off[kWgMaxBlocks], mul_in[kWgMaxBlocks], mul_out[kWgMaxBlocks], dim[kWgMaxBlocks],
      w_off[kWgMaxBlocks];
  double scale[kWgMaxBlocks];
  int32_t cta_begin[kWgMaxBlocks + 1];
  int in_dim, out_dim, S, splits;
  const void* x;
  const void* g;
  const int32_t* sperm;
  const int32_t* sptr;
  void* part;  // [splits][weight_numel]
  int64_t numel;
  int64_t N;
};

// CTA <-> (block b, species s, u tile, w tile, split): partial dW tile over the split's node range.
// The (u, w) tile is at most 64 x 64 but follows the block (the l = 2 irreps have 4 output channels): a thread owns
// 4 x 4 outputs, tun x tcn threads cover the tile, and the remaining threads form KG - 1 more "row groups" that take
// every KG-th staged row; the row groups are summed in a fixed order at the end (deterministic).
template <typename T>
__global__ void __launch_bounds__(256) linear_wgrad_kernel(const WgParams p) {
  __shared__ __align__(16) T smem_w[2 * kWgRows * (kWgTile + 1)];
  T(*xs)[kWgTile + 1] = reinterpret_cast<T(*)[kWgTile + 1]>(smem_w);
  T(*gs)[kWgTile + 1] = reinterpret_cast<T(*)[kWgTile + 1]>(smem_w + kWgRows * (kWgTile + 1));
  int b = 0;
  while (b + 1 < p.num_blocks && (int)blockIdx.x >= p.cta_begin[b + 1]) ++b;
  int local = blockIdx.x - p.cta_begin[b];
  const int mi = p.mul_in[b], mo = p.mul_out[b], d = p.dim[b];
  const int ut = ceil_div<int>(mi, kWgTile), wt = ceil_div<int>(mo, kWgTile);
  const int split = local % p.splits; local /= p.splits;
  const int wti = local % wt; local /= wt;
  const int uti = local % ut; local /= ut;
  const int s = local;
  int64_t lo = 0, hi = p.N;
  if (p.sptr) { lo = p.sptr[s]; hi = p.sptr[s + 1]; }
  const int64_t cnt = hi - lo;
  const int64_t n_begin = lo + cnt * split / p.splits, n_end = lo + cnt * (split + 1) / p.splits;
  const int u0 = uti * kWgTile, w0 = wti * kWgTile;
  const int nu = min(kWgTile, mi - u0), nw = min(kWgTile, mo - w0);
  const int tun = (nu + 3) >> 2, tcn = (nw + 3) >> 2;  // threads along u / w
  const int per = tun * tcn;
  const int KG = 256 / per;                            // row groups (per <= 256)
  const int tid = threadIdx.x;
  const int kg = tid / per, rem = tid - kg * per;
  const int tu = rem / tcn, tw = rem - tu * tcn;
  const bool active = kg < KG;
  const T* __restrict__ X = static_cast<const T*>(p.x);
  const T* __restrict__ G = static_cast<const T*>(p.g);
  using P = typename pair_of<T>::type;  // column pairs: one FFMA2 per pair in fp32
  P acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) acc[i][j].x = acc[i][j].y = T(0);
  const int npt = max(1, kWgRows / d);  // nodes per step (rows = nodes x d <= kWgRows: d <= 9)
  for (int64_t nb = n_begin; nb < n_end; nb += npt) {
    const int tn = (int)imin64(npt, n_end - nb);
    __syncthreads();
    for (int t = tid; t < kWgRows * kWgTile; t += blockDim.x) {
      const int r = t / kWgTile, c = t - r * kWgTile;
      const int j = r / d, m = r - j * d;
      T xv = T(0), gv = T(0);
      if (j < tn) {
        const int64_t node = p.sperm ? p.sperm[nb + j] : (nb + j);
        if (c < nu) xv = X[(size_t)node * p.in_dim + p.in_off[b] + (u0 + c) * d + m];
        if (c < nw) gv = G[(size_t)node * p.out_dim + p.out_off[b] + (w0 + c) * d + m];
      }
      xs[r][c] = xv;
      gs[r][c] = gv;
    }
    __syncthreads();
    const int rows = tn * d;
    if (active) {
      for (int r = kg; r < rows; r += KG) {
        T a[4], bb[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = xs[r][tu * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) bb[j] = gs[r][tw * 4 + j];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          fma_pair(a[i], bb[0], bb[1], acc[i][0]);
          fma_pair(a[i], bb[2], bb[3], acc[i][1]);
        }
      }
    }
  }
  // fixed-order sum over the row groups: red[kg][output] aliases the staging buffers (<= 256 x 16 elements)
  __syncthreads();
  T* red = smem_w;
  if (active) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        red[(size_t)kg * per * 16 + rem * 16 + i * 4 + j] = (j & 1) ? acc[i][j >> 1].y : acc[i][j >> 1].x;
  }
  __syncthreads();
  const T scale = T(p.scale[b]);
  T* part = static_cast<T*>(p.part) + (size_t)split * p.numel;
  for (int t = tid; t < per * 16; t += blockDim.x) {
    const int rm = t >> 4, ij = t & 15;
    const int tu2 = rm / tcn, tw2 = rm - tu2 * tcn;
    const int ul = tu2 * 4 + (ij >> 2), wl = tw2 * 4 + (ij & 3);
    if (ul >= nu || wl >= nw) continue;
    T sum = T(0);
    for (int q = 0; q < KG; ++q) sum += red[(size_t)q * per * 16 + t];
    part[(size_t)p.w_off[b] + ((size_t)(u0 + ul) * p.S + s) * mo + (w0 + wl)] = sum * scale;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) sum_partials_kernel(const T* __restrict__ part, int64_t stride, int nparts,
                                                           int64_t count, int accumulate, T* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= count) return;
  T s = accumulate ? out[i] : T(0);
  for (int b = 0; b < nparts; ++b) s += part[(size_t)b * stride + i];
  out[i] = s;
}

// --------------------------------------------------------------------------------------------- gate
template <typename T>
__global__ void __launch_bounds__(256) gate_bwd_kernel(const T* __restrict__ x, const T* __restrict__ g, int in_dim,
                                                       int out_dim, const int32_t* __restrict__ src_idx,
                                                       const int32_t* __restrict__ gate_idx,
                                                       const int32_t* __restrict__ act_id,
                                                       const T* __restrict__ act_cst, const T* __restrict__ aff_a,
                                                       const int32_t* __restrict__ inv_first,
                                                       const int32_t* __restrict__ inv_count, T* __restrict__ dx,
                                                       int64_t N) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= N * in_dim) return;
  const int64_t n = t / in_dim;
  const int i = (int)(t - n * in_dim);
  const T* xr = x + n * in_dim;
  const T* gr = g + n * out_dim;
  const int cnt = inv_count[i];
  T r = T(0);
  if (cnt > 0) {
    const int j0 = inv_first[i];
    if (src_idx[j0] == i) {
      // scalar (gate_idx < 0) or gated element: exactly one output
      T gv = gr[j0];
      if (aff_a) gv *= aff_a[j0];
      const int gi = gate_idx[j0];
      if (gi < 0) r = gv * apply_act_grad<T>(act_id[j0], xr[i]) * act_cst[j0];
      else r = gv * apply_act<T>(act_id[j0], xr[gi]) * act_cst[j0];
    } else {
      // a gate: feeds the cnt gated outputs j0 .. j0 + cnt - 1
      T s = T(0);
      for (int q = 0; q < cnt; ++q) {
        T gv = gr[j0 + q];
        if (aff_a) gv *= aff_a[j0 + q];
        s = fma(gv, xr[src_idx[j0 + q]], s);
      }
      r = s * apply_act_grad<T>(act_id[j0], xr[i]) * act_cst[j0];
    }
  }
  dx[t] = r;
}

// ------------------------------------------------------------------------------------ column reductions
constexpr int kColParts = 256;

template <typename T>
__global__ void __launch_bounds__(256) col_reduce_kernel(const T* __restrict__ a, const T* __restrict__ sa,
                                                         const T* __restrict__ b, const T* __restrict__ sb, int64_t N,
                                                         int dim, T* __restrict__ part) {
  const int64_t rows_per = ceil_div<int64_t>(N, (int64_t)gridDim.x);
  const int64_t r0 = blockIdx.x * rows_per, r1 = imin64(r0 + rows_per, N);
  for (int j = threadIdx.x; j < dim; j += blockDim.x) {
    const T va = sa ? sa[j] : T(0), vb = sb ? sb[j] : T(0);
    T s = T(0);
    if (b) {
      for (int64_t r = r0; r < r1; ++r) s = fma(a[r * dim + j] - va, b[r * dim + j] - vb, s);
    } else {
      for (int64_t r = r0; r < r1; ++r) s += a[r * dim + j] - va;
    }
    part[(size_t)blockIdx.x * dim + j] = s;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) affine2_kernel(const T* __restrict__ a, const T* __restrict__ ca,
                                                      const T* __restrict__ b, const T* __restrict__ cb,
                                                      const T* __restrict__ cc, T* __restrict__ out, int64_t N, int dim) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= N * dim) return;
  const int j = (int)(t % dim);
  T v = ca[j] * a[t];
  if (b) v = fma(cb[j], b[t], v);
  if (cc) v += cc[j];
  out[t] = v;
}

// ------------------------------------------------------------------------------------------ pooling
template <typename T>
__global__ void __launch_bounds__(256) segment_reduce_bwd_kernel(const T* __restrict__ g, const int32_t* __restrict__ ptr,
                                                                 int dim, int64_t B, int64_t N, int mode,
                                                                 T* __restrict__ dx) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= N * dim) return;
  const int64_t n = t / dim;
  const int j = (int)(t - n * dim);
  // largest b with ptr[b] <= n
  int64_t lo = 0, hi = B;
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (ptr[mid] <= n) lo = mid; else hi = mid;
  }
  T v = g[lo * dim + j];
  if (mode == 1) v = v / T(ptr[lo + 1] - ptr[lo]);
  dx[t] = v;
}

// thread <-> (segment, column): serial fixed-order sum (short segments)
template <typename T>
__global__ void __launch_bounds__(256) segment_sum_gather_kernel(const T* __restrict__ x, const int32_t* __restrict__ perm,
                                                                 const int32_t* __restrict__ ptr, int dim, int64_t S,
                                                                 T* __restrict__ out) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= S * dim) return;
  const int64_t s = t / dim;
  const int j = (int)(t - s * dim);
  const int i0 = ptr[s], i1 = ptr[s + 1];
  T acc = T(0);
  for (int i = i0; i < i1; ++i) {
    const int64_t r = perm ? perm[i] : i;
    acc += x[r * dim + j];
  }
  out[t] = acc;
}

// CTA <-> (segment, 32 columns): 8 warps stride the rows, fixed-order tree over the warps (long segments)
template <typename T>
__global__ void __launch_bounds__(256) segment_sum_gather_long_kernel(const T* __restrict__ x,
                                                                      const int32_t* __restrict__ perm,
                                                                      const int32_t* __restrict__ ptr, int dim,
                                                                      T* __restrict__ out) {
  __shared__ T red[8][33];
  const int s = blockIdx.x, j = blockIdx.y * 32 + (threadIdx.x & 31), w = threadIdx.x >> 5;
  const int i0 = ptr[s], i1 = ptr[s + 1];
  T acc = T(0);
  if (j < dim)
    for (int i = i0 + w; i < i1; i += 8) {
      const int64_t r = perm ? perm[i] : i;
      acc += x[r * dim + j];
    }
  red[w][threadIdx.x & 31] = acc;
  __syncthreads();
  if (w == 0 && j < dim) {
    T v = red[0][threadIdx.x];
#pragma unroll
    for (int q = 1; q < 8; ++q) v += red[q][threadIdx.x];
    out[(size_t)s * dim + j] = v;
  }
}

// ------------------------------------------------------------------------------------- loss / optimiser
template <typename T>
__global__ void __launch_bounds__(1024) mse_loss_kernel(const T* __restrict__ pred, const T* __restrict__ target,
                                                        int64_t n, T grad_scale, T* __restrict__ loss,
                                                        T* __restrict__ grad) {
  __shared__ T red[1024];
  T s = T(0);
  const T inv_n = T(1) / T(n);
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const T d = pred[i] - target[i];
    s = fma(d, d, s);
    if (grad) grad[i] = T(2) * d * inv_n * grad_scale;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int off = 512; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0 && loss) loss[0] = red[0] * inv_n;
}

template <typename T>
__global__ void __launch_bounds__(256) adam_step_kernel(T* __restrict__ p, const T* __restrict__ g, T* __restrict__ m,
                                                        T* __restrict__ v, int64_t n, T lr, T b1, T b2, T eps, T wd,
                                                        T grad_scale, T bc1, T bc2_sqrt) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T pi = p[i];
  const T gi = fma(wd, pi, g[i] * grad_scale);
  const T mi = fma(b1, m[i], (T(1) - b1) * gi);
  const T vi = fma(b2, v[i], (T(1) - b2) * gi * gi);
  m[i] = mi;
  v[i] = vi;
  const T denom = sqrt(vi) / bc2_sqrt + eps;
  p[i] = pi - (lr / bc1) * (mi / denom);
}

}  // namespace mt

using namespace mt;

extern "C" {

size_t mt_linear_bwd_workspace_bytes(int dtype, int64_t weight_numel) {
  return (size_t)wg_max_splits(weight_numel) * (size_t)weight_numel * (dtype == MT_F64 ? 8 : 4);
}

int mt_linear_bwd(int dtype, const mt_lin_block* blocks, int num_blocks, int in_dim, int out_dim, int num_species,
                  int64_t weight_numel, const void* x, const void* weight, const void* grad_out,
                  const int32_t* species_perm, const int32_t* species_ptr, void* grad_x, int accumulate_x,
                  void* grad_w, int accumulate_w, void* workspace, size_t workspace_bytes, int64_t N,
                  mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(blocks && num_blocks > 0 && num_blocks <= kWgMaxBlocks, "num_blocks %d not in 1..%d", num_blocks,
             kWgMaxBlocks);
  MT_REQUIRE(in_dim > 0 && out_dim > 0 && num_species >= 1, "bad dims");
  MT_REQUIRE((species_perm == nullptr) == (species_ptr == nullptr), "species_perm/ptr must be given together");
  MT_REQUIRE(num_species == 1 || species_ptr != nullptr, "species grouping required when num_species > 1");
  int rc = linear_check_blocks(blocks, num_blocks, in_dim, out_dim, weight, grad_x != nullptr);
  if (rc != MT_OK) return rc;
  cudaStream_t st = as_stream(stream);
  const size_t es = dtype == MT_F64 ? 8 : 4;
  if (N == 0) {
    if (grad_w && !accumulate_w) MT_CUDA_OK(cudaMemsetAsync(grad_w, 0, (size_t)weight_numel * es, st));
    return MT_OK;
  }
  MT_REQUIRE(grad_out != nullptr, "null grad_out");
  if (grad_x) {
    rc = linear_transposed(dtype, blocks, num_blocks, in_dim, out_dim, num_species, grad_out, weight, species_perm,
                           species_ptr, accumulate_x, grad_x, N, st);
    if (rc != MT_OK) return rc;
  }
  if (grad_w) {
    MT_REQUIRE(x != nullptr, "null x");
    MT_REQUIRE(workspace && workspace_bytes >= mt_linear_bwd_workspace_bytes(dtype, weight_numel),
               "linear_bwd workspace too small");
    WgParams p;
    memset(&p, 0, sizeof(p));
    int nb = 0;
    int64_t per_species = N / num_species;
    // a species-free linear over 3e4 nodes with 16 splits is 32 CTAs on 148 SMs (1.2 ms for the head's hidden layer):
    // small weights take up to 128 node ranges
    int splits = (int)(per_species / 256);
    if (splits < 1) splits = 1;
    if (splits > wg_max_splits(weight_numel)) splits = wg_max_splits(weight_numel);
    int64_t total = 0;
    for (int b = 0; b < num_blocks; ++b) {
      const mt_lin_block& k = blocks[b];
      if (k.mul_in == 0) continue;
      p.in_off[nb] = k.in_off; p.out_off[nb] = k.out_off; p.mul_in[nb] = k.mul_in; p.mul_out[nb] = k.mul_out;
      p.dim[nb] = k.dim; p.w_off[nb] = k.w_off;
      p.scale[nb] = k.scale;
      p.cta_begin[nb] = (int32_t)total;
      total += (int64_t)num_species * ceil_div<int>(k.mul_in, kWgTile) * ceil_div<int>(k.mul_out, kWgTile) * splits;
      ++nb;
    }
    p.cta_begin[nb] = (int32_t)total;
    MT_REQUIRE(total < (int64_t)2147483647, "grid too large");
    p.num_blocks = nb;
    p.in_dim = in_dim; p.out_dim = out_dim; p.S = num_species; p.splits = splits;
    p.x = x; p.g = grad_out; p.sperm = species_perm; p.sptr = species_ptr;
    p.part = workspace; p.numel = weight_numel; p.N = N;
    if (nb > 0) {
      // elements of weights whose block was skipped do not exist (mul_in == 0 -> no weights): every element of the
      // partial buffers is written by exactly one CTA
      MT_DISPATCH_DTYPE(dtype, { linear_wgrad_kernel<T><<<(unsigned)total, 256, 0, st>>>(p); });
      MT_LAUNCH_OK();
      MT_DISPATCH_DTYPE(dtype, {
        sum_partials_kernel<T><<<(unsigned)ceil_div<int64_t>(weight_numel, 256), 256, 0, st>>>(
            static_cast<const T*>(workspace), weight_numel, splits, weight_numel, accumulate_w, static_cast<T*>(grad_w));
      });
      MT_LAUNCH_OK();
    } else if (!accumulate_w) {
      MT_CUDA_OK(cudaMemsetAsync(grad_w, 0, (size_t)weight_numel * es, st));
    }
  }
  return MT_OK;
}

int mt_gate_bwd(int dtype, const void* x, const void* grad_out, int in_dim, int out_dim, const int32_t* src_idx,
                const int32_t* gate_idx, const int32_t* act_id, const void* act_cst, const void* affine_a,
                const int32_t* inv_first, const int32_t* inv_count, void* grad_x, int64_t N, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(in_dim > 0 && out_dim > 0, "bad dims");
  if (N == 0) return MT_OK;
  MT_REQUIRE(x && grad_out && grad_x && src_idx && gate_idx && act_id && act_cst && inv_first && inv_count,
             "null pointer");
  const int64_t total = N * in_dim;
  MT_DISPATCH_DTYPE(dtype, {
    gate_bwd_kernel<T><<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, as_stream(stream)>>>(
        (const T*)x, (const T*)grad_out, in_dim, out_dim, src_idx, gate_idx, act_id, (const T*)act_cst,
        (const T*)affine_a, inv_first, inv_count, (T*)grad_x, N);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

size_t mt_col_reduce_workspace_bytes(int dtype, int dim) {
  return (size_t)kColParts * (size_t)dim * (dtype == MT_F64 ? 8 : 4);
}

int mt_col_reduce(int dtype, const void* a, const void* shift_a, const void* b, const void* shift_b, int64_t N,
                  int dim, void* out, void* workspace, size_t workspace_bytes, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(dim > 0 && out != nullptr, "bad arguments");
  cudaStream_t st = as_stream(stream);
  const size_t es = dtype == MT_F64 ? 8 : 4;
  if (N == 0) {
    MT_CUDA_OK(cudaMemsetAsync(out, 0, (size_t)dim * es, st));
    return MT_OK;
  }
  MT_REQUIRE(a != nullptr, "null pointer");
  MT_REQUIRE(workspace && workspace_bytes >= mt_col_reduce_workspace_bytes(dtype, dim), "col_reduce workspace too small");
  int parts = (int)(N < kColParts ? N : kColParts);
  MT_DISPATCH_DTYPE(dtype, {
    col_reduce_kernel<T><<<parts, 256, 0, st>>>((const T*)a, (const T*)shift_a, (const T*)b, (const T*)shift_b, N, dim,
                                                (T*)workspace);
  });
  MT_LAUNCH_OK();
  MT_DISPATCH_DTYPE(dtype, {
    sum_partials_kernel<T><<<(unsigned)ceil_div<int>(dim, 256), 256, 0, st>>>((const T*)workspace, dim, parts, dim, 0,
                                                                             (T*)out);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_affine2(int dtype, const void* a, const void* ca, const void* b, const void* cb, const void* cc, void* out,
               int64_t N, int dim, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(dim > 0, "bad dim");
  if (N == 0) return MT_OK;
  MT_REQUIRE(a && ca && out && ((b == nullptr) == (cb == nullptr)), "null pointer");
  const int64_t total = N * dim;
  MT_DISPATCH_DTYPE(dtype, {
    affine2_kernel<T><<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, as_stream(stream)>>>(
        (const T*)a, (const T*)ca, (const T*)b, (const T*)cb, (const T*)cc, (T*)out, N, dim);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_segment_reduce_bwd(int dtype, const void* grad_out, const int32_t* ptr, int dim, int64_t B, int64_t N,
                          int mode, void* grad_x, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(dim > 0 && (mode == 0 || mode == 1), "segment_reduce_bwd supports sum and mean");
  if (N == 0) return MT_OK;
  MT_REQUIRE(grad_out && ptr && grad_x && B > 0, "null pointer");
  const int64_t total = N * dim;
  MT_DISPATCH_DTYPE(dtype, {
    segment_reduce_bwd_kernel<T><<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, as_stream(stream)>>>(
        (const T*)grad_out, ptr, dim, B, N, mode, (T*)grad_x);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_segment_sum_gather(int dtype, const void* x, const int32_t* perm, const int32_t* ptr, int dim,
                          int64_t num_segments, int64_t num_rows, void* out, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(dim > 0 && num_segments >= 0 && num_rows >= 0, "bad arguments");
  if (num_segments == 0) return MT_OK;
  MT_REQUIRE(ptr && out && (num_rows == 0 || x), "null pointer");
  cudaStream_t st = as_stream(stream);
  if (num_rows / num_segments >= 256 && num_segments <= 65535) {
    dim3 grid((unsigned)num_segments, (unsigned)ceil_div<int>(dim, 32));
    MT_DISPATCH_DTYPE(dtype, {
      segment_sum_gather_long_kernel<T><<<grid, 256, 0, st>>>((const T*)x, perm, ptr, dim, (T*)out);
    });
  } else {
    const int64_t total = num_segments * dim;
    MT_DISPATCH_DTYPE(dtype, {
      segment_sum_gather_kernel<T><<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, st>>>(
          (const T*)x, perm, ptr, dim, num_segments, (T*)out);
    });
  }
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_mse_loss(int dtype, const void* pred, const void* target, int64_t n, double grad_scale, void* loss, void* grad,
                mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(n > 0 && pred && target, "bad arguments");
  MT_DISPATCH_DTYPE(dtype, {
    mse_loss_kernel<T><<<1, 1024, 0, as_stream(stream)>>>((const T*)pred, (const T*)target, n, T(grad_scale), (T*)loss,
                                                          (T*)grad);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_adam_step(int dtype, void* p, const void* g, void* m, void* v, int64_t n, double lr, double beta1, double beta2,
                 double eps, double weight_decay, double grad_scale, int64_t step, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(n >= 0 && step >= 1, "bad arguments");
  if (n == 0) return MT_OK;
  MT_REQUIRE(p && g && m && v, "null pointer");
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2s = sqrt(1.0 - pow(beta2, (double)step));
  MT_DISPATCH_DTYPE(dtype, {
    adam_step_kernel<T><<<(unsigned)ceil_div<int64_t>(n, 256), 256, 0, as_stream(stream)>>>(
        (T*)p, (const T*)g, (T*)m, (T*)v, n, T(lr), T(beta1), T(beta2), T(eps), T(weight_decay), T(grad_scale), T(bc1),
        T(bc2s));
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

}  // extern "C"
