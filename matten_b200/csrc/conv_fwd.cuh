// Fused  radial-MLP -> uvu Clebsch-Gordan tensor product -> segmented sum over the
// receiver's edges  (rows a6 + a7 of SURVEY.md section 8).
//
// Replaces, for one PointConv layer, the chain of reference
//   src/matten/nn/utils.py:260   weight = weight_nn(edge_embedding)        [E, W]
//   src/matten/nn/utils.py:263   msg = tp(x[src], sh, weight)              [E, D_mid]
//   src/matten/nn/conv.py:114    scatter(msg, dst, dim_size=N)             atomics
//   src/matten/nn/conv.py:116    .div(avg_num_neighbors ** 0.5)
// Neither the per-edge weights nor the messages ever exist in HBM.
//
// Work decomposition (v1, FP32/FP64 FMA pipes):
//   CTA   <-> a tile of consecutive receiver nodes; its edges are a contiguous range of
//             the receiver-sorted edge list and are staged through shared memory in
//             chunks of <= EC edges: gathered sender rows x[src], sh rows, and the
//             hidden activations of the radial MLP (computed in the CTA).
//   warp  <-> one "item" (32 weight columns of one (l1,l2,l3) type) x one node.
//   lane  <-> one column (path p, channel u): holds its column of the last MLP layer
//             in registers, walks the node's edges, forms w[e,p,u] (H FMAs), runs the
//             unrolled CG contraction and accumulates the node's output in registers.
//   The per-node sum is a register accumulation in CSR order: deterministic, no atomics.
//   Types with fewer than 32 columns split the node's edges over lane groups
//   ("phases") and finish with a fixed-order shuffle reduction.
// HP == 0 is the variant for radial MLPs wider than 64 (radial_mlp.cuh): the per-edge weights are read from
// ConvFwdParams::wpe [E][Wn] (lanes hold consecutive columns: coalesced) instead of being formed from the staged
// hidden activations; there is no embedding staging and no hidden layer.
#pragma once
#include "common.cuh"
#include "generated/cg_gen.cuh"

namespace mt {

struct ConvFwdParams {
  int x_dim, y_dim, out_dim, num_items;
  const int32_t* item_hdr;
  const int32_t* slot_tab;
  int nl;  // number of MLP weight matrices
  int sizes[MT_MAX_MLP_LAYERS + 1];
  int act;
  double act_cst;
  const void* w[MT_MAX_MLP_LAYERS];
  const void* x;
  const void* sh;
  const void* emb;
  const int32_t* rowptr;
  const int32_t* perm;
  const int32_t* src;
  double avg;
  const void* num_neigh;
  void* out;
  int64_t N, E;
  int tile_nodes;   // receiver nodes per CTA tile
  int chunk_edges;  // EC
  int xs_stride;    // smem row stride of staged x rows
  int hp_max;       // smem row stride of the hidden-activation buffers
  const void* wpe;  // HP == 0: per-edge weights [E][sizes[nl]], receiver-sorted order
};

template <typename T>
__device__ __forceinline__ void load4(const T* p, T (&v)[4]);
template <>
__device__ __forceinline__ void load4<float>(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void load4<double>(const double* p, double (&v)[4]) {
  double2 a = *reinterpret_cast<const double2*>(p);
  double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// One warp, one item, one node: walk the node's staged edges [el0, el1).
// HP == 0: hs points at the lane's column of the chunk's first per-edge weight row, hstride = Wn.
template <typename T, int HP, int L1, int L2, int L3>
__device__ __forceinline__ void conv_unit(const T (&wreg)[HP > 0 ? HP : 1], const T* __restrict__ hs, int hstride,
                                          const T* __restrict__ xs, int xstride,
                                          const T* __restrict__ ys, int ystride, int xoff, int yoff,
                                          int el0, int el1, int phase, int nphase, int cpw,
                                          T* __restrict__ o, T den, bool first, bool do_write) {
  constexpr int D1 = 2 * L1 + 1, D2 = 2 * L2 + 1, D3 = 2 * L3 + 1;
  T acc[D3];
#pragma unroll
  for (int m = 0; m < D3; ++m) acc[m] = T(0);
  for (int el = el0 + phase; el < el1; el += nphase) {
    T w;
    if constexpr (HP == 0) {
      w = hs[(size_t)el * hstride];
    } else {
      const T* h = hs + (size_t)el * hstride;
      T w0 = T(0), w1 = T(0);
#pragma unroll
      for (int k = 0; k < HP; k += 8) {
        T a[4], b[4];
        load4<T>(h + k, a);
        load4<T>(h + k + 4, b);
        w0 = fma(a[0], wreg[k + 0], w0);
        w1 = fma(b[0], wreg[k + 4], w1);
        w0 = fma(a[1], wreg[k + 1], w0);
        w1 = fma(b[1], wreg[k + 5], w1);
        w0 = fma(a[2], wreg[k + 2], w0);
        w1 = fma(b[2], wreg[k + 6], w1);
        w0 = fma(a[3], wreg[k + 3], w0);
        w1 = fma(b[3], wreg[k + 7], w1);
      }
      w = w0 + w1;
    }
    T xv[D1], yv[D2];
    const T* xr = xs + (size_t)el * xstride + xoff;
#pragma unroll
    for (int m = 0; m < D1; ++m) xv[m] = xr[m];
    const T* yr = ys + (size_t)el * ystride + yoff;
#pragma unroll
    for (int m = 0; m < D2; ++m) yv[m] = yr[m];
    CG<L1, L2, L3>::template fwd<T>(xv, yv, w, acc);
  }
  // fixed-order reduction over the edge phases (lanes l, l+cpw, l+2cpw, ...)
  for (int off = cpw; off < 32; off <<= 1) {
#pragma unroll
    for (int m = 0; m < D3; ++m) acc[m] += __shfl_xor_sync(0xffffffffu, acc[m], off);
  }
  if (do_write) {
#pragma unroll
    for (int m = 0; m < D3; ++m) {
      const T v = acc[m] / den;  // true division, like torch's .div()
      o[m] = first ? v : (o[m] + v);
    }
  }
}

// resident CTAs per SM the register budget is compiled for
template <typename T, int HP>
__host__ __device__ constexpr int conv_fwd_min_blocks() {
  return sizeof(T) == 4 ? (HP <= 32 ? 3 : 2) : 1;
}

template <typename T, int HP>
__global__ void __launch_bounds__(256, (conv_fwd_min_blocks<T, HP>())) conv_fwd_kernel(const ConvFwdParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int EC = p.chunk_edges;
  T* ha = reinterpret_cast<T*>(smem_raw);
  T* hb = ha + (size_t)EC * p.hp_max;
  T* xs = hb + (size_t)EC * p.hp_max;
  T* ys = xs + (size_t)EC * p.xs_stride;
  T* wh = ys + (size_t)EC * p.y_dim;  // hidden-layer weights, pre-scaled by 1/sqrt(fan_in)
  __shared__ int s_counter;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const T* __restrict__ X = static_cast<const T*>(p.x);
  const T* __restrict__ SH = static_cast<const T*>(p.sh);
  const T* __restrict__ EMB = static_cast<const T*>(p.emb);
  T* __restrict__ OUT = static_cast<T*>(p.out);
  const int H_last = p.sizes[p.nl - 1];
  const T* __restrict__ Wlast = static_cast<const T*>(p.w[p.nl - 1]);
  const int Wn = p.sizes[p.nl];
  const T inv_sqrt_h = T(1) / sqrt(T(H_last));

  if constexpr (HP > 0) {
    int off = 0;
    for (int li = 0; li + 1 < p.nl; ++li) {
      const int fi = p.sizes[li], fo = p.sizes[li + 1];
      const T* __restrict__ Wl = static_cast<const T*>(p.w[li]);
      const T s = T(1) / sqrt(T(fi));
      for (int t = threadIdx.x; t < fi * fo; t += blockDim.x) wh[off + t] = Wl[t] * s;
      off += fi * fo;
    }
  }
  __syncthreads();

  const int64_t num_tiles = ceil_div<int64_t>(p.N, p.tile_nodes);
  for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int64_t n0 = tile * p.tile_nodes;
    const int tn = (int)imin64(p.tile_nodes, p.N - n0);
    const int e_begin = p.rowptr[n0], e_end = p.rowptr[n0 + tn];
    int c0 = e_begin;
    do {
      const int c1 = min(c0 + EC, e_end);
      const int ne = c1 - c0;
      // ------------------------------------------------------------ staging
      // gathered sender rows: one warp per edge row, coalesced
      for (int el = warp; el < ne; el += nwarps) {
        const T* xr = X + (size_t)p.src[c0 + el] * p.x_dim;
        T* xd = xs + (size_t)el * p.xs_stride;
        for (int j = lane; j < p.x_dim; j += 32) xd[j] = xr[j];
      }
      for (int t = tid; t < ne * p.y_dim; t += blockDim.x) {
        int el = t / p.y_dim, j = t - el * p.y_dim;
        ys[t] = SH[(size_t)p.perm[c0 + el] * p.y_dim + j];
      }
      if constexpr (HP > 0) {
        const int in0 = p.sizes[0];
        for (int t = tid; t < ne * p.hp_max; t += blockDim.x) {
          int el = t / p.hp_max, j = t - el * p.hp_max;
          ha[t] = (j < in0) ? EMB[(size_t)p.perm[c0 + el] * in0 + j] : T(0);
        }
      }
      if (tid == 0) s_counter = 0;
      __syncthreads();
      // hidden layers of the radial MLP: act(h @ W / sqrt(fan_in)) * cst
      T* hin = ha;
      T* hout = hb;
      int woff = 0;
      for (int li = 0; HP > 0 && li + 1 < p.nl; ++li) {
        const int fi = p.sizes[li], fo = p.sizes[li + 1];
        const T* Wl = wh + woff;
        woff += fi * fo;
        const T cst = T(p.act_cst);
        for (int t = tid; t < ne * p.hp_max; t += blockDim.x) {
          int el = t / p.hp_max, j = t - el * p.hp_max;
          T v = T(0);
          if (j < fo) {
            const T* hr = hin + (size_t)el * p.hp_max;
            T a = T(0);
            for (int k = 0; k < fi; ++k) a = fma(hr[k], Wl[k * fo + j], a);
            v = apply_act<T>(p.act, a) * cst;
          }
          hout[t] = v;
        }
        __syncthreads();
        T* tmp = hin; hin = hout; hout = tmp;
      }
      const T* hs = hin;  // [ne][hp_max], zero padded beyond H_last

      // ------------------------------------------------------------ compute
      const int num_units = p.num_items * tn;
      while (true) {
        int unit = 0;
        if (lane == 0) unit = atomicAdd(&s_counter, 1);
        unit = __shfl_sync(0xffffffffu, unit, 0);
        if (unit >= num_units) break;
        const int item = unit / tn;
        const int nl_ = unit - item * tn;
        const int64_t n = n0 + nl_;
        const int type = p.item_hdr[item * 2 + 0];
        const int cpw = p.item_hdr[item * 2 + 1];
        const int4 slot = reinterpret_cast<const int4*>(p.slot_tab)[item * 32 + lane];
        const int wcol = slot.x, xoff = slot.y, yoff = slot.z, ooff = slot.w;
        const int phase = lane / cpw, nphase = 32 / cpw;
        T wreg[HP > 0 ? HP : 1];
#pragma unroll
        for (int k = 0; k < HP; ++k)
          wreg[k] = (wcol >= 0 && k < H_last) ? Wlast[(size_t)k * Wn + wcol] * inv_sqrt_h : T(0);
        const int r0 = p.rowptr[n], r1 = p.rowptr[n + 1];
        const int lo = max(r0, c0), hi = min(r1, c1);
        const bool first = (r0 >= c0) || (c0 == e_begin);
        if (lo >= hi && !(r0 == r1 && c0 == e_begin)) continue;  // nothing for this node in this chunk
        const T den = p.num_neigh ? sqrt(static_cast<const T*>(p.num_neigh)[n]) : sqrt(T(p.avg));
        T* o = OUT + (size_t)n * p.out_dim + ooff;
        const bool do_write = (wcol >= 0) && (phase == 0);
        if constexpr (HP == 0) {
          // idle lanes (wcol < 0) read column 0 and write nothing
          const T* wsrc = static_cast<const T*>(p.wpe) + (size_t)c0 * Wn + (wcol >= 0 ? wcol : 0);
          switch (type) {
#define MT_CONV_CASE(ID, A, B, C)                                                                   \
  case ID:                                                                                          \
    conv_unit<T, HP, A, B, C>(wreg, wsrc, Wn, xs, p.xs_stride, ys, p.y_dim, xoff, yoff, lo - c0,     \
                              hi - c0, phase, nphase, cpw, o, den, first, do_write);                \
    break;
            MT_FOR_EACH_CG_TYPE(MT_CONV_CASE)
#undef MT_CONV_CASE
            default: break;
          }
        } else {
          switch (type) {
#define MT_CONV_CASE(ID, A, B, C)                                                                   \
  case ID:                                                                                          \
    conv_unit<T, HP, A, B, C>(wreg, hs, p.hp_max, xs, p.xs_stride, ys, p.y_dim, xoff, yoff, lo - c0, \
                              hi - c0, phase, nphase, cpw, o, den, first, do_write);                \
    break;
            MT_FOR_EACH_CG_TYPE(MT_CONV_CASE)
#undef MT_CONV_CASE
            default: break;
          }
        }
      }
      __syncthreads();
      c0 += EC;
    } while (c0 < e_end);
  }
}

}  // namespace mt
