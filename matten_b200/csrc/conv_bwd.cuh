// Backward of the fused convolution (mt_conv_bwd, include/matten_b200.h).
//
// What autograd does in the reference through
//   src/matten/nn/utils.py:260   weight = weight_nn(edge_embedding)
//   src/matten/nn/utils.py:263   msg = tp(x[src], sh, weight)
//   src/matten/nn/conv.py:114    scatter(msg, dst)        conv.py:116  .div(sqrt(avg_num_neighbors))
// restated as five kernels, none of which materialises the messages:
//   K0 edge_hidden_kernel      pre-activations z_l of the hidden MLP layers per edge (receiver-sorted order)
//   K1 conv_bwd_kernel         CTA <-> tile of receiver nodes, edges staged in shared memory in chunks:
//                              (A) per-edge weights w[e,:] = a_last[e,:] @ W_last/sqrt(H) into shared memory,
//                              (B) warp <-> (32 input channels of one irrep) x node, lane <-> channel u: walks
//                                  the node's edges and, per edge, every path reading the channel:
//                                  dw[e,c] = <CG(x_u, Y), g_u>/den -> DW scratch; dx_u += w[e,c]/den * CG^T(Y, g_u)
//                                  -> DXE scratch.  Register sums in fixed path order: deterministic.
//   K2 mlp_bwd_last_kernel     dW_last = a_last^T DW / sqrt(H) (per-CTA partials) and da_last = DW W_last^T/sqrt(H)
//   K3 mlp_bwd_hidden_kernel   the hidden layers: dz = da * act'(z) * cst, dW_l partials, da_l
//   K4 reduce_partials_kernel  fixed-order sum of the per-CTA partial weight gradients
// and the per-sender sum of DXE rows over the sender CSR (segment_sum_gather, node_ops.cu).
//
// Gradients with respect to the edge inputs (mt_conv_bwd_full), in separate instantiations so that the plain backward
// keeps its code:
//   grad_sh   conv_bwd_kernel<T, true>: in phase B every lane also forms CG^T(x_u, g_u) w for the sh components of
//             each path, reduced over the unit's channels by a fixed shuffle tree into one partial row per
//             (item, staged edge) in shared memory; after phase B the rows are summed over the items in item order.
//   grad_emb  dz0 W0^T / sqrt(fan_in) in K3 (both forms), or the column-group sum of K2's da_last for a one-layer MLP.
// Both are written through perm (a permutation) in the caller's edge order.
#pragma once
#include "common.cuh"
#include "generated/cg_gen.cuh"

namespace mt {

constexpr int kBwdMaxH = 64;     // largest MLP layer input/hidden size the backward supports
constexpr int kBwdET = 8;        // edges per register pass of phase A (chunk_edges is a multiple of it)
constexpr int kLastEB = 64;      // edges per chunk of K2
constexpr int kLastCW = 128;     // weight columns per CTA column group of K2
constexpr int kHidEBMax = 64;    // edges per chunk of K0 / K3 (halved until the tiles fit: ConvBwdParams::hid_eb)

struct ConvBwdParams {
  int x_dim, y_dim, out_dim, Wn;
  int num_items, num_paths;
  const int32_t* item_hdr;  // [num_items][4]
  const int32_t* lane_tab;  // [num_items][32][2]
  const int32_t* path_tab;  // [num_paths][4]
  int nl;
  int sizes[MT_MAX_MLP_LAYERS + 1];
  int act;
  double act_cst;
  const void* w[MT_MAX_MLP_LAYERS];
  void* z[MT_MAX_MLP_LAYERS];  // z[l] [E][sizes[l+1]] for l < nl-1 (workspace)
  const void* x;
  const void* sh;
  const void* emb;
  const int32_t* rowptr;
  const int32_t* perm;
  const int32_t* src;
  double avg;
  const void* num_neigh;
  const void* g;   // grad_out [N][out_dim]
  void* DW;        // [E][Wn]
  void* DXE;       // [E][x_dim]
  void* DHP;       // [ncg][E][H]
  void* PARTL;     // [grid2][H][Wn]
  void* PARTH;     // [grid3][hidden numel]
  int64_t N, E;
  int tile_nodes, chunk_edges, xs_stride, hs_stride, wt_stride;
  int ncg, grid2, grid3, hid_numel;
  int hid_eb;  // edges per chunk of K0 / K3
  int rs;  // row stride of the per-edge activation tiles of K0 / K3: largest input / hidden size + 1
  void* gsh;   // [E][y_dim] gradient w.r.t. sh (original edge order), written by conv_bwd_kernel<T, true>
  void* gemb;  // [E][sizes[0]] gradient w.r.t. the edge embedding (original edge order)
};

template <typename T>
__device__ __forceinline__ void load4(const T* p, T (&v)[4]);
template <>
__device__ __forceinline__ void load4<float>(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void load4<double>(const double* p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// last-layer input a_{nl-1}[e][k]: act(z_{nl-2}) * cst, or the embedding itself for a single-layer MLP
template <typename T>
__device__ __forceinline__ T last_input(const ConvBwdParams& p, int64_t e, int k) {
  if (p.nl == 1) return static_cast<const T*>(p.emb)[(size_t)p.perm[e] * p.sizes[0] + k];
  const T z = static_cast<const T*>(p.z[p.nl - 2])[(size_t)e * p.sizes[p.nl - 1] + k];
  return apply_act<T>(p.act, z) * T(p.act_cst);
}

// ---------------------------------------------------------------------------------------------- K0
template <typename T>
__global__ void __launch_bounds__(256) edge_hidden_kernel(const ConvBwdParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int RS = p.rs, EB = p.hid_eb;
  T* A = reinterpret_cast<T*>(smem_raw);               // [EB][RS]
  T* Wl = A + (size_t)EB * RS;                     // [<=64][<=64] of the current layer, pre-scaled
  const int tid = threadIdx.x;
  const int64_t nchunks = ceil_div<int64_t>(p.E, EB);
  for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int64_t e0 = ch * EB;
    const int ne = (int)imin64(EB, p.E - e0);
    const int in0 = p.sizes[0];
    __syncthreads();
    for (int t = tid; t < ne * in0; t += blockDim.x) {
      const int el = t / in0, k = t - el * in0;
      A[el * RS + k] = static_cast<const T*>(p.emb)[(size_t)p.perm[e0 + el] * in0 + k];
    }
    for (int l = 0; l + 1 < p.nl; ++l) {
      const int fi = p.sizes[l], fo = p.sizes[l + 1];
      const T s = T(1) / sqrt(T(fi));
      const T* __restrict__ Wg = static_cast<const T*>(p.w[l]);
      for (int t = tid; t < fi * fo; t += blockDim.x) Wl[t] = Wg[t] * s;
      __syncthreads();
      T* Z = static_cast<T*>(p.z[l]);
      for (int t = tid; t < ne * fo; t += blockDim.x) {
        const int el = t / fo, j = t - el * fo;
        const T* ar = A + el * RS;
        T acc = T(0);
        for (int k = 0; k < fi; ++k) acc = fma(ar[k], Wl[k * fo + j], acc);
        Z[(size_t)(e0 + el) * fo + j] = acc;
      }
      __syncthreads();
      // every thread re-reads the entries it wrote itself (same t mapping): no fence needed
      for (int t = tid; t < ne * fo; t += blockDim.x) {
        const int el = t / fo, j = t - el * fo;
        A[el * RS + j] = apply_act<T>(p.act, Z[(size_t)(e0 + el) * fo + j]) * T(p.act_cst);
      }
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------------------------------------- K1
// bwd_unit with the sh gradient: every lane of the warp runs the same trip count (idle lanes and lanes past the last
// edge compute nothing and contribute zeros), so that the per-path sh partials can be summed over the cpw lanes of a
// phase by a fixed xor-shuffle tree; the phase's first lane adds them to the (item, edge) row ysp[el][:] in path order.
template <typename T, int L1>
__device__ __forceinline__ void bwd_unit_eg(const ConvBwdParams& p, const int4* __restrict__ spath, int pfirst,
                                            int pcount, int u, int xoff, const T* __restrict__ xs,
                                            const T* __restrict__ ys, const T* __restrict__ wt,
                                            const T* __restrict__ gs, const int* __restrict__ enode,
                                            const T* __restrict__ sden, int el0, int el1, int phase, int nphase,
                                            int c0, T* __restrict__ ysp) {
  constexpr int D1 = 2 * L1 + 1;
  T* __restrict__ DW = static_cast<T*>(p.DW);
  T* __restrict__ DXE = static_cast<T*>(p.DXE);
  const int cpw = 32 / nphase;
  const bool leader = (threadIdx.x & (cpw - 1)) == 0;
  const bool lane_on = u >= 0;
  const int uu = lane_on ? u : 0;  // idle lanes read channel 0 (xoff is 0 for them) and discard the result
  for (int base = el0; base < el1; base += nphase) {
    const int el = base + phase;
    const bool live = el < el1;
    const bool on = lane_on && live;
    const int elc = live ? el : el0;
    T xv[D1], dxv[D1];
    const T* xr = xs + (size_t)elc * p.xs_stride + xoff;
#pragma unroll
    for (int m = 0; m < D1; ++m) { xv[m] = xr[m]; dxv[m] = T(0); }
    const T* wrow = wt + (size_t)elc * p.wt_stride;
    const T* yrow = ys + (size_t)elc * p.y_dim;
    const int nl_ = enode[elc];
    const T* gn = gs + (size_t)nl_ * p.out_dim;
    const T inv_den = sden[nl_];
    T* dwrow = DW + (size_t)(c0 + elc) * p.Wn;
    T* yp = ysp + (size_t)elc * p.y_dim;
    for (int pk = 0; pk < pcount; ++pk) {
      const int4 pt = spath[pfirst + pk];
      const int c = pt.y + uu;
      const T w = wrow[c] * inv_den;
      switch (pt.x) {
#define MT_CONV_BWD_EG_CASE(ID, A, B, C)                                           \
  case ID:                                                                    \
    if constexpr (A == L1) {                                                  \
      constexpr int D2 = 2 * B + 1, D3 = 2 * C + 1;                           \
      T yv[D2], gv[D3], dy[D2];                                               \
      _Pragma("unroll") for (int m = 0; m < D2; ++m) { yv[m] = yrow[pt.z + m]; dy[m] = T(0); } \
      const T* gr = gn + pt.w + uu * D3;                                      \
      _Pragma("unroll") for (int m = 0; m < D3; ++m) gv[m] = gr[m];           \
      if (on) {                                                               \
        dwrow[c] = CG<A, B, C>::template dot<T>(xv, yv, gv) * inv_den;        \
        CG<A, B, C>::template bwd_x<T>(yv, gv, w, dxv);                       \
        CG<A, B, C>::template bwd_y<T>(xv, gv, w, dy);                        \
      }                                                                       \
      for (int o = cpw >> 1; o > 0; o >>= 1)                                  \
        _Pragma("unroll") for (int m = 0; m < D2; ++m) dy[m] += __shfl_xor_sync(0xffffffffu, dy[m], o); \
      if (leader && live)                                                     \
        _Pragma("unroll") for (int m = 0; m < D2; ++m) yp[pt.z + m] += dy[m]; \
    }                                                                         \
    break;
        MT_FOR_EACH_CG_TYPE(MT_CONV_BWD_EG_CASE)
#undef MT_CONV_BWD_EG_CASE
        default: break;
      }
    }
    if (on) {
      T* dxr = DXE + (size_t)(c0 + el) * p.x_dim + xoff;
#pragma unroll
      for (int m = 0; m < D1; ++m) dxr[m] = dxv[m];
    }
  }
}

template <typename T, int L1, bool EG>
__device__ __forceinline__ void bwd_unit(const ConvBwdParams& p, const int4* __restrict__ spath, int pfirst, int pcount,
                                         int u, int xoff, const T* __restrict__ xs, const T* __restrict__ ys,
                                         const T* __restrict__ wt, const T* __restrict__ gs,
                                         const int* __restrict__ enode, const T* __restrict__ sden, int el0, int el1,
                                         int phase, int nphase, int c0, T* __restrict__ ysp) {
  constexpr int D1 = 2 * L1 + 1;
  T* __restrict__ DW = static_cast<T*>(p.DW);
  T* __restrict__ DXE = static_cast<T*>(p.DXE);
  if constexpr (EG) {
    bwd_unit_eg<T, L1>(p, spath, pfirst, pcount, u, xoff, xs, ys, wt, gs, enode, sden, el0, el1, phase, nphase, c0, ysp);
    return;
  }
  if (u < 0) return;
  for (int el = el0 + phase; el < el1; el += nphase) {
    T xv[D1], dxv[D1];
    const T* xr = xs + (size_t)el * p.xs_stride + xoff;
#pragma unroll
    for (int m = 0; m < D1; ++m) { xv[m] = xr[m]; dxv[m] = T(0); }
    const T* wrow = wt + (size_t)el * p.wt_stride;
    const T* yrow = ys + (size_t)el * p.y_dim;
    const int nl_ = enode[el];  // receiver of this edge within the tile
    const T* gn = gs + (size_t)nl_ * p.out_dim;
    const T inv_den = sden[nl_];
    T* dwrow = DW + (size_t)(c0 + el) * p.Wn;
    for (int pk = 0; pk < pcount; ++pk) {
      const int4 pt = spath[pfirst + pk];  // {type, weight column of u = 0, sh offset, out offset of u = 0}
      const int c = pt.y + u;
      const T w = wrow[c] * inv_den;
      switch (pt.x) {
#define MT_CONV_BWD_CASE(ID, A, B, C)                                   \
  case ID:                                                         \
    if constexpr (A == L1) {                                       \
      constexpr int D2 = 2 * B + 1, D3 = 2 * C + 1;                \
      T yv[D2], gv[D3];                                            \
      _Pragma("unroll") for (int m = 0; m < D2; ++m) yv[m] = yrow[pt.z + m]; \
      const T* gr = gn + pt.w + u * D3;                            \
      _Pragma("unroll") for (int m = 0; m < D3; ++m) gv[m] = gr[m]; \
      dwrow[c] = CG<A, B, C>::template dot<T>(xv, yv, gv) * inv_den; \
      CG<A, B, C>::template bwd_x<T>(yv, gv, w, dxv);              \
    }                                                              \
    break;
        MT_FOR_EACH_CG_TYPE(MT_CONV_BWD_CASE)
#undef MT_CONV_BWD_CASE
        default: break;
      }
    }
    T* dxr = DXE + (size_t)(c0 + el) * p.x_dim + xoff;
#pragma unroll
    for (int m = 0; m < D1; ++m) dxr[m] = dxv[m];
  }
}

template <typename T, bool EG>
__global__ void __launch_bounds__(256, sizeof(T) == 4 ? 3 : 2) conv_bwd_kernel(const ConvBwdParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int EC = p.chunk_edges;
  int4* spath = reinterpret_cast<int4*>(smem_raw);     // [num_paths]
  T* hs = reinterpret_cast<T*>(spath + p.num_paths);   // [hs_stride >= H][EC] transposed last-layer input
  T* xs = hs + (size_t)EC * p.hs_stride;               // [EC][xs_stride]
  T* ys = xs + (size_t)EC * p.xs_stride;               // [EC][y_dim]
  T* wt = ys + (size_t)EC * p.y_dim;                   // [EC][wt_stride]
  T* gs = wt + (size_t)EC * p.wt_stride;               // [tile_nodes][out_dim]
  T* sden = gs + (size_t)p.tile_nodes * p.out_dim;     // [tile_nodes] 1 / sqrt(#neighbours)
  int* enode = reinterpret_cast<int*>(sden + p.tile_nodes);  // [EC] receiver (tile-local) of every staged edge
  T* ysp = reinterpret_cast<T*>(enode + EC);  // EG: [num_items][EC][y_dim] sh-gradient partials (EC % 8 == 0: aligned)
  __shared__ int s_counter;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const T* __restrict__ X = static_cast<const T*>(p.x);
  const T* __restrict__ SH = static_cast<const T*>(p.sh);
  const T* __restrict__ G = static_cast<const T*>(p.g);
  const int H = p.sizes[p.nl - 1];
  const T* __restrict__ Wlast = static_cast<const T*>(p.w[p.nl - 1]);
  const int Wn = p.Wn;
  const T inv_sqrt_h = T(1) / sqrt(T(H));

  for (int t = tid; t < p.num_paths; t += blockDim.x) spath[t] = reinterpret_cast<const int4*>(p.path_tab)[t];
  __syncthreads();

  const int64_t num_tiles = ceil_div<int64_t>(p.N, p.tile_nodes);
  for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int64_t n0 = tile * p.tile_nodes;
    const int tn = (int)imin64(p.tile_nodes, p.N - n0);
    const int e_begin = p.rowptr[n0], e_end = p.rowptr[n0 + tn];
    if (e_begin == e_end) continue;
    __syncthreads();
    // grad_out rows of the tile's nodes
    for (int t = tid; t < tn * p.out_dim; t += blockDim.x) gs[t] = G[(size_t)n0 * p.out_dim + t];
    for (int t = tid; t < tn; t += blockDim.x) {
      const T den = p.num_neigh ? sqrt(static_cast<const T*>(p.num_neigh)[n0 + t]) : sqrt(T(p.avg));
      sden[t] = T(1) / den;
    }
    for (int c0 = e_begin; c0 < e_end; c0 += EC) {
      const int c1 = min(c0 + EC, e_end);
      const int ne = c1 - c0;
      __syncthreads();
      // ------------------------------------------------------------ staging
      for (int el = warp; el < ne; el += nwarps) {
        const T* xr = X + (size_t)p.src[c0 + el] * p.x_dim;
        T* xd = xs + (size_t)el * p.xs_stride;
        for (int j = lane; j < p.x_dim; j += 32) xd[j] = xr[j];
      }
      for (int t = tid; t < ne * p.y_dim; t += blockDim.x) {
        const int el = t / p.y_dim, j = t - el * p.y_dim;
        ys[t] = SH[(size_t)p.perm[c0 + el] * p.y_dim + j];
      }
      // a_last / sqrt(H), TRANSPOSED [k][EC] so that the 8 edges of a register pass are one 128-bit broadcast load
      for (int t = tid; t < EC * H; t += blockDim.x) {
        const int k = t / EC, el = t - k * EC;  // lanes walk the edges: conflict-free stores
        hs[(size_t)k * EC + el] = (el < ne) ? last_input<T>(p, (int64_t)c0 + el, k) * inv_sqrt_h : T(0);
      }
      for (int el = tid; el < ne; el += blockDim.x) {
        int j = 0;
        while (j + 1 < tn && p.rowptr[n0 + j + 1] <= c0 + el) ++j;
        enode[el] = j;
      }
      if constexpr (EG)
        for (int t = tid; t < p.num_items * EC * p.y_dim; t += blockDim.x) ysp[t] = T(0);
      if (tid == 0) s_counter = 0;
      __syncthreads();
      // ------------------------------------------------------------ (A) per-edge weights into shared memory
      // register tile: 8 edges x 2 columns (c, c + blockDim) per thread
      for (int ep = 0; ep < ne; ep += kBwdET) {
        for (int c = tid; c < Wn; c += 2 * blockDim.x) {
          const int c2 = c + blockDim.x;
          const bool two = c2 < Wn;
          using P = typename pair_of<T>::type;  // edge pairs: one FFMA2 (broadcast weight) per pair in fp32
          P acc0[kBwdET / 2], acc1[kBwdET / 2];
#pragma unroll
          for (int i = 0; i < kBwdET / 2; ++i) { acc0[i].x = acc0[i].y = T(0); acc1[i].x = acc1[i].y = T(0); }
#pragma unroll 4
          for (int k = 0; k < H; ++k) {
            const T w0 = Wlast[(size_t)k * Wn + c];
            const T w1 = two ? Wlast[(size_t)k * Wn + c2] : T(0);
            T hv[kBwdET];
            load4<T>(hs + (size_t)k * EC + ep, *reinterpret_cast<T(*)[4]>(&hv[0]));
            load4<T>(hs + (size_t)k * EC + ep + 4, *reinterpret_cast<T(*)[4]>(&hv[4]));
#pragma unroll
            for (int i = 0; i < kBwdET / 2; ++i) {
              fma_pair(w0, hv[2 * i], hv[2 * i + 1], acc0[i]);
              fma_pair(w1, hv[2 * i], hv[2 * i + 1], acc1[i]);
            }
          }
#pragma unroll
          for (int i = 0; i < kBwdET; ++i)
            if (ep + i < ne) {
              wt[(size_t)(ep + i) * p.wt_stride + c] = (i & 1) ? acc0[i >> 1].y : acc0[i >> 1].x;
              if (two) wt[(size_t)(ep + i) * p.wt_stride + c2] = (i & 1) ? acc1[i >> 1].y : acc1[i >> 1].x;
            }
        }
      }
      __syncthreads();
      // ------------------------------------------------------------ (B) units: (item, block of 8 staged edges).
      // The outputs are per edge, so a unit need not be a whole node: small units keep the 8 warps balanced.
      const int nblk = (ne + 7) >> 3;
      const int num_units = p.num_items * nblk;
      while (true) {
        int unit = 0;
        if (lane == 0) unit = atomicAdd(&s_counter, 1);
        unit = __shfl_sync(0xffffffffu, unit, 0);
        if (unit >= num_units) break;
        const int item = unit / nblk;
        const int eb = unit - item * nblk;
        const int4 hdr = reinterpret_cast<const int4*>(p.item_hdr)[item];  // {l1, cpw, first path, count}
        const int2 ls = reinterpret_cast<const int2*>(p.lane_tab)[item * 32 + lane];
        const int cpw = hdr.y;
        const int phase = lane / cpw, nphase = 32 / cpw;
        const int lo = eb * 8, hi = min(lo + 8, ne);
        T* yspi = ysp + (size_t)item * EC * p.y_dim;
        switch (hdr.x) {
          case 0: bwd_unit<T, 0, EG>(p, spath, hdr.z, hdr.w, ls.x, ls.y, xs, ys, wt, gs, enode, sden, lo, hi, phase, nphase, c0, yspi); break;
          case 1: bwd_unit<T, 1, EG>(p, spath, hdr.z, hdr.w, ls.x, ls.y, xs, ys, wt, gs, enode, sden, lo, hi, phase, nphase, c0, yspi); break;
          case 2: bwd_unit<T, 2, EG>(p, spath, hdr.z, hdr.w, ls.x, ls.y, xs, ys, wt, gs, enode, sden, lo, hi, phase, nphase, c0, yspi); break;
          case 3: bwd_unit<T, 3, EG>(p, spath, hdr.z, hdr.w, ls.x, ls.y, xs, ys, wt, gs, enode, sden, lo, hi, phase, nphase, c0, yspi); break;
          case 4: bwd_unit<T, 4, EG>(p, spath, hdr.z, hdr.w, ls.x, ls.y, xs, ys, wt, gs, enode, sden, lo, hi, phase, nphase, c0, yspi); break;
          default: break;
        }
      }
      if constexpr (EG) {
        // grad_sh of the chunk's edges: the item partials summed in item order
        __syncthreads();
        T* GSH = static_cast<T*>(p.gsh);
        for (int t = tid; t < ne * p.y_dim; t += blockDim.x) {
          const int el = t / p.y_dim, j = t - el * p.y_dim;
          T s = T(0);
          for (int it = 0; it < p.num_items; ++it) s += ysp[((size_t)it * EC + el) * p.y_dim + j];
          GSH[(size_t)p.perm[c0 + el] * p.y_dim + j] = s;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- K2
// grid (grid2, ncg): CTA (bx, cg) walks edge chunks bx, bx + grid2, ... for the weight columns of group cg.
template <typename T, int HP>
__global__ void __launch_bounds__(256) mlp_bwd_last_kernel(const ConvBwdParams p) {
  constexpr int KP = HP / 8 > 0 ? HP / 8 : 1;  // k per thread of the dW tile (k = tk + 8 i)
  constexpr int KD = HP / 4;                   // k per thread of the dH tile
  constexpr int DS = kLastCW + 4;              // row stride of the dw tile
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* dws = reinterpret_cast<T*>(smem_raw);             // [kLastEB][DS]
  T* hs2 = dws + (size_t)kLastEB * DS;                 // [kLastEB][HP]
  T* WlT = hs2 + (size_t)kLastEB * HP;                 // [kLastCW][HP]  (pre-scaled by 1/sqrt(H))
  const int tid = threadIdx.x;
  const int H = p.sizes[p.nl - 1], Wn = p.Wn;
  const int cg = blockIdx.y;
  const int cbase = cg * kLastCW;
  const int ncol = min(kLastCW, Wn - cbase);
  const T inv_sqrt_h = T(1) / sqrt(T(H));
  const T* __restrict__ Wlast = static_cast<const T*>(p.w[p.nl - 1]);
  const T* __restrict__ DW = static_cast<const T*>(p.DW);
  for (int t = tid; t < kLastCW * HP; t += blockDim.x) {
    const int c = t / HP, k = t - c * HP;
    WlT[t] = (c < ncol && k < H) ? Wlast[(size_t)k * Wn + cbase + c] * inv_sqrt_h : T(0);
  }
  const int tc = tid & 31, tk = tid >> 5;   // dW tile: columns 4 tc .. 4 tc + 3, k = tk + 8 i
  const int te = tid >> 2, kq = tid & 3;    // dH tile: edge te, k = kq * KD .. + KD - 1
  using P = typename pair_of<T>::type;  // pairs of columns / of k: one FFMA2 per pair in fp32
  P accw[KP][2];
#pragma unroll
  for (int i = 0; i < KP; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) accw[i][j].x = accw[i][j].y = T(0);
  const int64_t nchunks = ceil_div<int64_t>(p.E, kLastEB);
  for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int64_t e0 = ch * kLastEB;
    const int ne = (int)imin64(kLastEB, p.E - e0);
    __syncthreads();
    for (int t = tid; t < kLastEB * kLastCW; t += blockDim.x) {
      const int el = t / kLastCW, c = t - el * kLastCW;
      dws[el * DS + c] = (el < ne && c < ncol) ? DW[(size_t)(e0 + el) * Wn + cbase + c] : T(0);
    }
    for (int t = tid; t < kLastEB * HP; t += blockDim.x) {
      const int el = t / HP, k = t - el * HP;
      hs2[t] = (el < ne && k < H) ? last_input<T>(p, e0 + el, k) : T(0);
    }
    __syncthreads();
    // dW_last[k][c] += sum_e a[e][k] dw[e][c]
    if (tk < HP) {
      for (int el = 0; el < kLastEB; ++el) {
        const T* dr = dws + el * DS + tc * 4;
        const T d0 = dr[0], d1 = dr[1], d2 = dr[2], d3 = dr[3];
#pragma unroll
        for (int i = 0; i < KP; ++i) {
          const T hv = hs2[el * HP + tk + 8 * i];
          fma_pair(hv, d0, d1, accw[i][0]);
          fma_pair(hv, d2, d3, accw[i][1]);
        }
      }
    }
    // dH[e][k] (this column group) = sum_c dw[e][c] W[k][c] / sqrt(H)
    {
      P acch[KD / 2];
#pragma unroll
      for (int i = 0; i < KD / 2; ++i) acch[i].x = acch[i].y = T(0);
      const T* dr = dws + te * DS;
      for (int c = 0; c < kLastCW; ++c) {
        const T dv = dr[c];
        const T* wr = WlT + c * HP + kq * KD;
#pragma unroll
        for (int i = 0; i < KD / 2; ++i) fma_pair(dv, wr[2 * i], wr[2 * i + 1], acch[i]);
      }
      if (te < ne) {
        T* dh = static_cast<T*>(p.DHP) + ((size_t)cg * p.E + (e0 + te)) * H;
#pragma unroll
        for (int i = 0; i < KD; ++i)
          if (kq * KD + i < H) dh[kq * KD + i] = (i & 1) ? acch[i >> 1].y : acch[i >> 1].x;
      }
    }
  }
  // partial dW_last of this CTA: PARTL[bx][k][c]
  T* part = static_cast<T*>(p.PARTL) + (size_t)blockIdx.x * H * Wn;
#pragma unroll
  for (int i = 0; i < KP; ++i) {
    const int k = tk + 8 * i;
    if (k < H) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = tc * 4 + j;
        if (c < ncol) part[(size_t)k * Wn + cbase + c] = (j & 1) ? accw[i][j >> 1].y : accw[i][j >> 1].x;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- K3
template <typename T, bool EMB>
__global__ void __launch_bounds__(256) mlp_bwd_hidden_kernel(const ConvBwdParams p) {
  const int RS = p.rs, EB = p.hid_eb;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* DA = reinterpret_cast<T*>(smem_raw);   // [EB][RS]  gradient w.r.t. the layer's output activation
  T* DZ = DA + (size_t)EB * RS;         // [EB][RS]
  T* A = DZ + (size_t)EB * RS;          // [EB][RS]  the layer's input activation
  T* Wl = A + (size_t)EB * RS;          // [<=64][fo + 1] current layer, pre-scaled (padded: lanes walk k)
  T* accW = Wl + (size_t)(RS - 1) * RS;     // [hid_numel] running partial sums of this CTA
  const int tid = threadIdx.x;
  for (int t = tid; t < p.hid_numel; t += blockDim.x) accW[t] = T(0);
  const int H = p.sizes[p.nl - 1];
  const int64_t nchunks = ceil_div<int64_t>(p.E, EB);
  for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int64_t e0 = ch * EB;
    const int ne = (int)imin64(EB, p.E - e0);
    __syncthreads();
    // da_{nl-1}: fixed-order sum of the column-group partials of K2
    for (int t = tid; t < EB * H; t += blockDim.x) {
      const int el = t / H, k = t - el * H;
      T s = T(0);
      if (el < ne)
        for (int cg = 0; cg < p.ncg; ++cg) s += static_cast<const T*>(p.DHP)[((size_t)cg * p.E + (e0 + el)) * H + k];
      DA[el * RS + k] = s;
    }
    int woff = p.hid_numel;
    for (int l = p.nl - 2; l >= 0; --l) {
      const int fi = p.sizes[l], fo = p.sizes[l + 1];
      woff -= fi * fo;
      const T s = T(1) / sqrt(T(fi));
      const T* __restrict__ Wg = static_cast<const T*>(p.w[l]);
      __syncthreads();
      for (int t = tid; t < fi * fo; t += blockDim.x) Wl[(t / fo) * (fo + 1) + (t % fo)] = Wg[t] * s;
      const T* Z = static_cast<const T*>(p.z[l]);
      for (int t = tid; t < EB * fo; t += blockDim.x) {
        const int el = t / fo, j = t - el * fo;
        T v = T(0);
        if (el < ne) v = DA[el * RS + j] * apply_act_grad<T>(p.act, Z[(size_t)(e0 + el) * fo + j]) * T(p.act_cst);
        DZ[el * RS + j] = v;
      }
      for (int t = tid; t < EB * fi; t += blockDim.x) {
        const int el = t / fi, k = t - el * fi;
        T v = T(0);
        if (el < ne) {
          if (l == 0) v = static_cast<const T*>(p.emb)[(size_t)p.perm[e0 + el] * fi + k];
          else v = apply_act<T>(p.act, static_cast<const T*>(p.z[l - 1])[(size_t)(e0 + el) * fi + k]) * T(p.act_cst);
        }
        A[el * RS + k] = v;
      }
      __syncthreads();
      // dW_l[k][j] += sum_e A[e][k] DZ[e][j]   (scaled by 1/sqrt(fi) in the final reduction)
      for (int t = tid; t < fi * fo; t += blockDim.x) {
        const int k = t / fo, j = t - k * fo;
        T acc = T(0);
        for (int el = 0; el < EB; ++el) acc = fma(A[el * RS + k], DZ[el * RS + j], acc);
        accW[woff + t] += acc;
      }
      __syncthreads();
      if (l > 0) {
        // da_l[e][k] = sum_j DZ[e][j] W_l[k][j] / sqrt(fi)
        for (int t = tid; t < EB * fi; t += blockDim.x) {
          const int el = t / fi, k = t - el * fi;
          T acc = T(0);
          for (int j = 0; j < fo; ++j) acc = fma(DZ[el * RS + j], Wl[k * (fo + 1) + j], acc);
          DA[el * RS + k] = acc;
        }
      } else if constexpr (EMB) {
        // grad_emb[e][k] = sum_j DZ[e][j] W_0[k][j] / sqrt(fi)
        for (int t = tid; t < ne * fi; t += blockDim.x) {
          const int el = t / fi, k = t - el * fi;
          T acc = T(0);
          for (int j = 0; j < fo; ++j) acc = fma(DZ[el * RS + j], Wl[k * (fo + 1) + j], acc);
          static_cast<T*>(p.gemb)[(size_t)p.perm[e0 + el] * fi + k] = acc;
        }
      }
    }
  }
  __syncthreads();
  T* part = static_cast<T*>(p.PARTH) + (size_t)blockIdx.x * p.hid_numel;
  for (int t = tid; t < p.hid_numel; t += blockDim.x) part[t] = accW[t];
}

// ---------------------------------------------------------------------------------------------- K0 / K3, fast forms
// The MLP shape of every matten config (n_rad <= 8 -> 32 -> 32 -> W, silu), fp32: lane == edge, a layer's 32 values in
// registers, weights by warp-wide broadcast LDS.128 (the generic kernels above walk [edge][k] tiles in shared memory
// with an integer division per element: 0.5 ms (K0) and 1.0 ms (K3) per layer at 9e5 edges against ~0.1 ms here).
__device__ __forceinline__ float bwd_sigmoid(float v) {  // ex2.approx + rcp.approx: ~3e-7 relative
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * v));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return r;
}

// y[0..31] += h * W[k][0..31] for a row of a [.][32] matrix in shared memory (broadcast LDS.128)
__device__ __forceinline__ void bwd_row_fma(float h, const float* __restrict__ wrow, float2 (&acc)[16]) {
  const float4* wr = reinterpret_cast<const float4*>(wrow);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 w = wr[j];
    fma_pair(h, w.x, w.y, acc[2 * j]);
    fma_pair(h, w.z, w.w, acc[2 * j + 1]);
  }
}

__global__ void __launch_bounds__(256) edge_hidden_fast_kernel(const ConvBwdParams p) {
  __shared__ __align__(16) float sW0[8 * 32];
  __shared__ __align__(16) float sW1[32 * 32];
  const int in0 = p.sizes[0];
  {
    const float s0 = rsqrtf((float)in0), s1 = rsqrtf(32.f);
    const float* w0 = static_cast<const float*>(p.w[0]);
    const float* w1 = static_cast<const float*>(p.w[1]);
    for (int t = threadIdx.x; t < 8 * 32; t += 256) sW0[t] = (t >> 5) < in0 ? w0[t] * s0 : 0.f;
    for (int t = threadIdx.x; t < 32 * 32; t += 256) sW1[t] = w1[t] * s1;
  }
  __syncthreads();
  const float cst = (float)p.act_cst;
  const float* __restrict__ emb = static_cast<const float*>(p.emb);
  float4* Z0 = static_cast<float4*>(p.z[0]);
  float4* Z1 = static_cast<float4*>(p.z[1]);
  for (int64_t e = blockIdx.x * 256ll + threadIdx.x; e < p.E; e += (int64_t)gridDim.x * 256) {
    const float* er = emb + (size_t)p.perm[e] * in0;
    float2 acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float h = k < in0 ? er[k] : 0.f;
      bwd_row_fma(h, sW0 + k * 32, acc);
    }
    float a1[32];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      Z0[(size_t)e * 8 + i] = make_float4(acc[2 * i].x, acc[2 * i].y, acc[2 * i + 1].x, acc[2 * i + 1].y);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      a1[2 * i] = acc[i].x * bwd_sigmoid(acc[i].x) * cst;
      a1[2 * i + 1] = acc[i].y * bwd_sigmoid(acc[i].y) * cst;
      acc[i] = make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < 32; ++k) bwd_row_fma(a1[k], sW1 + k * 32, acc);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      Z1[(size_t)e * 8 + i] = make_float4(acc[2 * i].x, acc[2 * i].y, acc[2 * i + 1].x, acc[2 * i + 1].y);
  }
}

// K3: one warp walks chunks of 32 edges (lane == edge).  Per chunk: da2 = sum of the K2 column-group partials,
// dz1 = da2 silu'(z1) cst, da1 = W1 dz1 / sqrt(32) (W1^T rows by broadcast LDS.128), dz0 = da1 silu'(z0) cst; then the
// chunk's a1 / dz1 and emb / dz0 go through warp-private shared-memory tiles and every lane accumulates one row of
// dW1 (lane == input index i: 32 sums in registers) and one column of dW0 (lane == output index j: 8 sums) over ALL
// its chunks.  One partial [hid_numel] per warp, summed in fixed order by reduce_partials_kernel.
constexpr int kHidFastWarps = 3;   // 3 x 13.6 KB of tiles + W1^T stay under the 48 KB static limit; 5 CTAs per SM
constexpr int kHidFastCtas = 5 * kNumSMs;
struct HidFastTile {
  float a1[32 * 33];   // [edge][i], stride 33: lane e writes row e, lane i reads column i -- both conflict free
  float dz0[32 * 33];  // [edge][j]
  float dz1[32 * 32];  // [edge][j] dense, float4 chunks XOR-swizzled by (edge & 7): broadcast LDS.128 reads
  float emb[32 * 8];   // [edge][k]
};

template <bool EMB>
__global__ void __launch_bounds__(32 * kHidFastWarps) mlp_bwd_hidden_fast_kernel(const ConvBwdParams p) {
  __shared__ __align__(16) float sW1T[32 * 32];  // [j][i] = W1[i][j] / sqrt(32)
  __shared__ __align__(16) HidFastTile tiles[kHidFastWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int in0 = p.sizes[0];
  {
    const float s1 = rsqrtf(32.f);
    const float* w1 = static_cast<const float*>(p.w[1]);
    for (int t = tid; t < 32 * 32; t += 32 * kHidFastWarps) sW1T[(t & 31) * 32 + (t >> 5)] = w1[t] * s1;
  }
  __syncthreads();
  HidFastTile& T = tiles[warp];
  const float cst = (float)p.act_cst;
  const float* __restrict__ emb = static_cast<const float*>(p.emb);
  const float4* Z0 = static_cast<const float4*>(p.z[0]);
  const float4* Z1 = static_cast<const float4*>(p.z[1]);
  const float4* DHP = static_cast<const float4*>(p.DHP);
  float2 gw1[16];  // dW1[lane][0..31]
  float2 gw0[4];   // dW0[0..7][lane]
#pragma unroll
  for (int i = 0; i < 16; ++i) gw1[i] = make_float2(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < 4; ++i) gw0[i] = make_float2(0.f, 0.f);
  const int64_t nchunks = (p.E + 31) >> 5;
  const int64_t wglobal = (int64_t)blockIdx.x * kHidFastWarps + warp, wtotal = (int64_t)gridDim.x * kHidFastWarps;
  for (int64_t ch = wglobal; ch < nchunks; ch += wtotal) {
    const int64_t e = ch * 32 + lane;
    const bool in = e < p.E;
    const int64_t es = in ? e : p.E - 1;  // lanes past the end compute on the last edge and contribute zeros
    // da2, dz1
    float dz1[32];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int cg = 0; cg < p.ncg; ++cg) {
        const float4 v = DHP[((size_t)cg * p.E + es) * 8 + i];
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      }
      const float4 z = Z1[(size_t)es * 8 + i];
      const float zz[4] = {z.x, z.y, z.z, z.w}, ss[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float sg = bwd_sigmoid(zz[q]);
        dz1[4 * i + q] = in ? ss[q] * (sg * (1.f + zz[q] * (1.f - sg))) * cst : 0.f;
      }
    }
    // da1 = W1 dz1 / sqrt(32)
    float2 da1[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) da1[i] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < 32; ++j) bwd_row_fma(dz1[j], sW1T + j * 32, da1);
    __syncwarp();  // the previous chunk's tiles have been consumed
#pragma unroll
    for (int i = 0; i < 8; ++i)
      *reinterpret_cast<float4*>(&T.dz1[lane * 32 + ((i ^ (lane & 7)) << 2)]) =
          make_float4(dz1[4 * i], dz1[4 * i + 1], dz1[4 * i + 2], dz1[4 * i + 3]);
    // a1, dz0 from z0; emb row
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 z = Z0[(size_t)es * 8 + i];
      const float zz[4] = {z.x, z.y, z.z, z.w};
      const float dd[4] = {da1[2 * i].x, da1[2 * i].y, da1[2 * i + 1].x, da1[2 * i + 1].y};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float sg = bwd_sigmoid(zz[q]);
        T.a1[lane * 33 + 4 * i + q] = in ? zz[q] * sg * cst : 0.f;
        T.dz0[lane * 33 + 4 * i + q] = in ? dd[q] * (sg * (1.f + zz[q] * (1.f - sg))) * cst : 0.f;
      }
    }
    if constexpr (EMB) {
      // grad_emb[e][k] = sum_j dz0[e][j] W0[k][j] / sqrt(in0)  (W0 rows by warp-uniform loads)
      const float* __restrict__ w0 = static_cast<const float*>(p.w[0]);
      const float s0 = rsqrtf((float)in0);
      float* ge = static_cast<float*>(p.gemb);
      for (int k = 0; k < in0; ++k) {
        float acc = 0.f;
#pragma unroll 8
        for (int j = 0; j < 32; ++j) acc = fmaf(T.dz0[lane * 33 + j], __ldg(w0 + k * 32 + j), acc);
        if (in) ge[(size_t)p.perm[e] * in0 + k] = acc * s0;
      }
    }
    {
      const float* er = emb + (size_t)p.perm[es] * in0;
#pragma unroll
      for (int k = 0; k < 8; ++k) T.emb[lane * 8 + k] = (in && k < in0) ? er[k] : 0.f;
    }
    __syncwarp();
    // dW1[lane][:] += sum_e a1[e][lane] dz1[e][:]     dW0[:][lane] += sum_e emb[e][:] dz0[e][lane]
#pragma unroll 4
    for (int el = 0; el < 32; ++el) {
      const float a = T.a1[el * 33 + lane];
      const float* dr = &T.dz1[el * 32];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 d = *reinterpret_cast<const float4*>(dr + ((i ^ (el & 7)) << 2));
        fma_pair(a, d.x, d.y, gw1[2 * i]);
        fma_pair(a, d.z, d.w, gw1[2 * i + 1]);
      }
      const float g0 = T.dz0[el * 33 + lane];
      const float4 e0 = *reinterpret_cast<const float4*>(&T.emb[el * 8]);
      const float4 e1 = *reinterpret_cast<const float4*>(&T.emb[el * 8 + 4]);
      fma_pair(g0, e0.x, e0.y, gw0[0]);
      fma_pair(g0, e0.z, e0.w, gw0[1]);
      fma_pair(g0, e1.x, e1.y, gw0[2]);
      fma_pair(g0, e1.z, e1.w, gw0[3]);
    }
  }
  // this warp's partial: layer 0 at [k][j] = k * 32 + j (k < in0), layer 1 at in0 * 32 + i * 32 + j
  float* part = static_cast<float*>(p.PARTH) + (size_t)wglobal * p.hid_numel;
  const float g0v[8] = {gw0[0].x, gw0[0].y, gw0[1].x, gw0[1].y, gw0[2].x, gw0[2].y, gw0[3].x, gw0[3].y};
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (k < in0) part[k * 32 + lane] = g0v[k];
  float4* p1 = reinterpret_cast<float4*>(part + in0 * 32 + lane * 32);
#pragma unroll
  for (int i = 0; i < 8; ++i) p1[i] = make_float4(gw1[2 * i].x, gw1[2 * i].y, gw1[2 * i + 1].x, gw1[2 * i + 1].y);
}

// grad_emb of a one-layer MLP (the embedding is the last layer's input): the fixed-order sum of K2's column-group
// partials of da_last, written through perm.
template <typename T>
__global__ void __launch_bounds__(256) emb_grad_last_kernel(const ConvBwdParams p) {
  const int H = p.sizes[0];
  const T* __restrict__ DHP = static_cast<const T*>(p.DHP);
  for (int64_t t = blockIdx.x * 256ll + threadIdx.x; t < p.E * H; t += (int64_t)gridDim.x * 256) {
    const int64_t e = t / H;
    const int k = (int)(t - e * H);
    T s = T(0);
    for (int cg = 0; cg < p.ncg; ++cg) s += DHP[((size_t)cg * p.E + e) * H + k];
    static_cast<T*>(p.gemb)[(size_t)p.perm[e] * H + k] = s;
  }
}

// ---------------------------------------------------------------------------------------------- K4
// CTA <-> 32 outputs x 8 partial groups: thread (o, g) sums partials g, g + 8, ... in order, the 8 group sums are then
// added in order -- a fixed summation tree (deterministic) with 8 x the memory parallelism of one serial loop per output.
template <typename T>
__global__ void __launch_bounds__(256) reduce_partials_kernel(const T* __restrict__ part, int64_t stride, int nparts,
                                                              int64_t off, int64_t count, T scale,
                                                              T* __restrict__ out) {
  __shared__ T sh[8][33];
  const int o = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int64_t i = blockIdx.x * 32ll + o;
  T s = T(0);
  if (i < count)
    for (int b = g; b < nparts; b += 8) s += part[(size_t)b * stride + off + i];
  sh[g][o] = s;
  __syncthreads();
  if (g == 0 && i < count) {
    T t = sh[0][o];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += sh[k][o];
    out[i] = t * scale;
  }
}

}  // namespace mt
