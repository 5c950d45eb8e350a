// Node-side kernels: species-indexed irreps linear (a8/a11/a13/a14), Gate + BatchNorm
// affine (a9/a10), segmented pooling (a12).  See include/matten_b200.h for the contract.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace mt {

// =========================================================================
// irreps-wise (species-indexed) linear
//   reference: e3nn FullyConnectedTensorProduct(x, one_hot, out) at
//   src/matten/nn/conv.py:59-61,77-79,84-86 and e3nn.o3.Linear at
//   src/matten/nn/nodewise.py:111.  With one-hot attributes the "uvw" tensor product is
//   a per-species dense matrix per irrep type; nodes are grouped by species so each CTA
//   applies ONE species' [mul_in x mul_out] weight slices, staged in shared memory, to a tile of its nodes.
//
// Node-streaming: one CTA owns a tile of nodes of ONE species and walks ALL irrep blocks over it.
//   * the species' weight slices of every block sit in shared memory for the CTA's lifetime;
//   * each block's input columns of the tile's rows arrive by cp.async (16 B per lane, coalesced along the row), one
//     block ahead of the arithmetic, so x is read from HBM exactly once and never passes through registers;
//   * lanes <-> output channels w, NB nodes per lane in registers: per 4 input channels a lane issues 4 LDS.32 of
//     weights (conflict free), NB x D LDS.128 of x (warp-wide broadcast) and NB x 4 x D FMAs.
// The round-1 tiled kernel spent 152 k thread instructions per node on lin2 of the last layer for 14.8 k MACs (rows
// of 1392 floats cut into 80-byte slivers per k-chunk, every chunk paying the DRAM latency): ncu r2_step_full.
// Two pipelines share that arithmetic: linear_sync_kernel (CTA-synchronous tiles, short rows) and
// linear_stream_kernel (warp-private, rows of >= 512 elements).  Blocks whose weight slice and rows fit neither in
// shared memory are cut into rectangles of their weight on the host (linear_apply).
// =========================================================================
constexpr int kLinMaxBlocks = 24;
constexpr int kStreamSmemBytes = 200 * 1024;

template <typename T>
__device__ __forceinline__ void lin_ld4(const T* p, T (&v)[4]);
template <>
__device__ __forceinline__ void lin_ld4<float>(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void lin_ld4<double>(const double* p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// one element global -> shared without passing through registers (LDGSTS); !valid zero-fills the destination
template <typename T>
__device__ __forceinline__ void lin_cp_async(T* smem_dst, const T* gsrc, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int n = valid ? (int)sizeof(T) : 0;
  if constexpr (sizeof(T) == 4)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}
__device__ __forceinline__ void lin_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void lin_cp_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct LinParams {
  int num_blocks;
  int32_t in_off[kLinMaxBlocks], out_off[kLinMaxBlocks], mul_in[kLinMaxBlocks], mul_out[kLinMaxBlocks],
      dim[kLinMaxBlocks], w_off[kLinMaxBlocks];
  // row stride of the weight: weight[w_off + (u * S + s) * ld + w] (transposed: [w_off + (w * S + s) * ld + u]).
  // ld is the mul_out (transposed: mul_in) of the whole block, also when the block is one piece of a cut.
  int32_t ld[kLinMaxBlocks];
  double scale[kLinMaxBlocks];
  int in_dim, out_dim, S;
  const void* x;
  const void* weight;
  const int32_t* sperm;
  const int32_t* sptr;
  int accumulate;
  int transpose;  // 1: apply the transposed weight slices (backward w.r.t. x): blocks come with in/out swapped
  void* out;
  int64_t N;
};

struct LinStream {
  int tnode;                        // nodes per CTA tile
  int rs;                           // row stride (elements) of the staged x rows: max over blocks, multiple of 4, + 4
  int w_smem_off[kLinMaxBlocks];    // element offset of block b's [mi4][mo] slice
  int w_total;                      // elements of all slices
  int vec_ok[kLinMaxBlocks];        // rows of this block can be copied 16 bytes at a time
  int w_vec[kLinMaxBlocks];         // ... and so can the rows of its weight slice
  int tiles_per_cta;                // consecutive tiles of one species per CTA (weights staged once for all of them)
};

// Each species' nodes are cut into tiles of `super` nodes, numbered species after species; CTA blockIdx.x takes one.
// false: a spare CTA (the grid counts a partial tile for every species).
__device__ __forceinline__ bool lin_locate(const LinParams& p, int super, int& s, int64_t& begin, int64_t& end) {
  int tile = blockIdx.x;
  s = 0;
  if (p.S == 1 && p.sptr == nullptr) {
    begin = (int64_t)tile * super;
    end = imin64(begin + super, p.N);
    return begin < p.N;
  }
  for (s = 0; s < p.S; ++s) {
    const int cnt = p.sptr[s + 1] - p.sptr[s];
    const int nt = (cnt + super - 1) / super;
    if (tile < nt) {
      begin = p.sptr[s] + (int64_t)tile * super;
      end = imin64(begin + super, (int64_t)p.sptr[s + 1]);
      return true;
    }
    tile -= nt;
  }
  return false;
}

// Species s's weight slices into shared memory, [mi4][mo] per block (rows mi..mi4 zero); asynchronous copies, all in
// flight at once, for the caller to commit as one group.  Rows of mo contiguous elements: 16 bytes per copy when mo
// allows.
template <typename T>
__device__ __forceinline__ void lin_stage_weights(const LinParams& p, const LinStream& e, T* wsm, int s) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const T* __restrict__ W = static_cast<const T*>(p.weight);
  constexpr int V = 16 / (int)sizeof(T);  // elements per 16-byte copy
  for (int b = 0; b < p.num_blocks; ++b) {
    const int mi = p.mul_in[b], mo = p.mul_out[b], ld = p.ld[b], mi4 = (mi + 3) & ~3;
    T* dst = wsm + e.w_smem_off[b];
    if (!p.transpose && e.w_vec[b]) {
      const int rowv = mo / V;  // vectors per row
      const int nvec = mi4 * rowv;
      int u = tid / rowv, c = tid - u * rowv;          // one division per thread and block; then additive
      const int du = 256 / rowv, dc = 256 - du * rowv;
      for (int v = tid; v < nvec; v += 256) {
        const bool ok = u < mi;
        const T* src = W + (ok ? (size_t)p.w_off[b] + ((size_t)u * p.S + s) * ld + c * V : 0);
        const uint32_t da = (uint32_t)__cvta_generic_to_shared(dst + u * mo + c * V);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(da), "l"(src), "r"(ok ? 16 : 0) : "memory");
        u += du; c += dc;
        if (c >= rowv) { c -= rowv; ++u; }
      }
    } else {
      for (int u = warp; u < mi4; u += 8)
        for (int w = lane; w < mo; w += 32) {
          const bool ok = u < mi;
          const size_t off = !ok ? 0
                             : p.transpose ? (size_t)p.w_off[b] + ((size_t)w * p.S + s) * ld + u
                                           : (size_t)p.w_off[b] + ((size_t)u * p.S + s) * ld + w;
          lin_cp_async<T>(dst + u * mo + w, W + off, ok);
        }
    }
  }
}

// One staged x row: the seg elements at src, then zeros up to segp (the padded length the arithmetic reads).  16 bytes
// per copy when the row is aligned (vec), else one element per copy.
template <typename T>
__device__ __forceinline__ void lin_stage_row(T* dst, const T* src, int seg, int segp, bool vec, int lane) {
  constexpr int V = 16 / (int)sizeof(T);  // elements per 16-byte copy
  if (vec) {
    const uint32_t drow = (uint32_t)__cvta_generic_to_shared(dst);
    for (int q = lane * V; q < segp; q += 32 * V) {
      const int n = min(V, seg - q);  // elements really there
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(drow + q * (int)sizeof(T)),
                   "l"(src + (n > 0 ? q : 0)), "r"(n > 0 ? n * (int)sizeof(T) : 0)
                   : "memory");
    }
  } else {
    for (int q = lane; q < segp; q += 32) lin_cp_async<T>(dst + q, src + (q < seg ? q : 0), q < seg);
  }
}

// lanes per output channel group: the smallest of 32/16/8/4 covering mul_out (32 when mul_out > 16)
__device__ __forceinline__ int lin_lpn(int mo) {
  int lpn = 32;
  while (lpn > 4 && (lpn >> 1) >= mo) lpn >>= 1;
  return lpn;
}

// One block for the output channels w0 .. w0 + lpn - 1 (lpn = lin_lpn(mo)) of NB nodes whose staged rows are
// xs + nb * RS, of which the first ncount are stored:
//   out[nodes[nb], out_off + w * D + m] (+)= scale * sum_u ws[u][w] * xs[nb][u * D + m].
// Lanes of a warp = (output channel w: lpn lanes) x (k-split ks: 32 / lpn lanes): every warp works on NB nodes
// whatever mul_out is; narrow outputs (mul_out 16 or 4 for l >= 1) split the input channels over the spare lanes and
// reduce with shuffles at the end.  The loops over w0 and over node groups stay in the kernels: the CTA-synchronous
// kernel runs node groups inside the w0 loop, and ptxas gives it fewer registers in that order.
template <typename T, int D, int NB>
__device__ __forceinline__ void lin_block(const T* __restrict__ ws, const T* __restrict__ xs, int RS, int mi4, int mo,
                                          int lpn, int w0, int ncount, const int* __restrict__ nodes,
                                          T* __restrict__ OUT, int out_dim, int out_off, T scale, int accumulate) {
  const int lane = threadIdx.x & 31;
  const int subs = 32 / lpn, ks = lane / lpn, wl = lane - ks * lpn;
  const int ustep = 4 * subs;
  const int w = w0 + wl;
  const bool wok = w < mo;
  T acc[NB][D];
  const T* xq[NB];
#pragma unroll
  for (int nb = 0; nb < NB; ++nb) {
#pragma unroll
    for (int m = 0; m < D; ++m) acc[nb][m] = T(0);
    // rows past ncount repeat the last one; never stored
    xq[nb] = xs + (size_t)min(nb, ncount - 1) * RS + ks * 4 * D;
  }
  const T* wq = ws + (wok ? w : 0) + ks * 4 * mo;
  for (int u = ks * 4; u < mi4; u += ustep) {
    T wv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) wv[k] = wq[k * mo];
    wq += ustep * mo;
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) {
      T xv[4 * D];
#pragma unroll
      for (int i = 0; i < D; ++i) lin_ld4<T>(xq[nb] + 4 * i, *reinterpret_cast<T(*)[4]>(&xv[4 * i]));
      xq[nb] += ustep * D;
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int m = 0; m < D; ++m) acc[nb][m] = fma(wv[k], xv[k * D + m], acc[nb][m]);
    }
  }
  for (int off = lpn; off < 32; off <<= 1) {  // sum the k-splits (fixed order: deterministic)
#pragma unroll
    for (int nb = 0; nb < NB; ++nb)
#pragma unroll
      for (int m = 0; m < D; ++m) acc[nb][m] += __shfl_xor_sync(0xffffffffu, acc[nb][m], off);
  }
  if (wok && ks == 0) {
#pragma unroll
    for (int nb = 0; nb < NB; ++nb) {
      if (nb < ncount) {
        T* dst = OUT + (size_t)nodes[nb] * out_dim + out_off + w * D;
#pragma unroll
        for (int m = 0; m < D; ++m) dst[m] = accumulate ? (dst[m] + acc[nb][m] * scale) : acc[nb][m] * scale;
      }
    }
  }
}

// CTA-synchronous variant (all warps walk the blocks together over a tile of 16 or 32 nodes, NB = 2 / 4 nodes per
// lane): better for the short rows of lin1 / sc, where amortising the weight loads over more nodes matters most.
constexpr int kStreamTiles = 8;  // at most: consecutive tiles of one species per CTA (weight slices staged once)

template <typename T>
__global__ void __launch_bounds__(256) linear_sync_kernel(const LinParams p, const LinStream e) {
  extern __shared__ __align__(16) unsigned char lin_smem[];
  __shared__ int s_nodes[kStreamTiles * 32];
  T* wsm = reinterpret_cast<T*>(lin_smem);
  T* xbuf = wsm + ((e.w_total + 3) & ~3);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int s;
  int64_t begin, end;
  if (!lin_locate(p, e.tnode * e.tiles_per_cta, s, begin, end)) return;
  const int tn_all = (int)(end - begin);
  const int ntiles = (tn_all + e.tnode - 1) / e.tnode;
  for (int i = tid; i < tn_all; i += 256) s_nodes[i] = p.sperm ? p.sperm[begin + i] : (int)(begin + i);
  const T* __restrict__ X = static_cast<const T*>(p.x);
  T* __restrict__ OUT = static_cast<T*>(p.out);
  lin_stage_weights<T>(p, e, wsm, s);  // the first group the pipeline below waits for
  lin_cp_commit();
  __syncthreads();  // s_nodes
  const int nb_ = p.num_blocks;
  const int nsteps = ntiles * nb_;
  auto issue = [&](int step) {
    const int t = step / nb_, b = step - t * nb_;
    const int mi = p.mul_in[b], d = p.dim[b];
    const int seg = mi * d, segp = (((mi + 3) & ~3) * d + 3) & ~3;  // copied + zero-filled up to the padded length
    const int n0 = t * e.tnode, tn = min(e.tnode, tn_all - n0);
    T* buf = xbuf + (size_t)(step & 1) * e.tnode * e.rs;
    if (mi > 0) {
      for (int j = warp; j < tn; j += 8)
        lin_stage_row<T>(buf + (size_t)j * e.rs, X + (size_t)s_nodes[n0 + j] * p.in_dim + p.in_off[b], seg, segp,
                         e.vec_ok[b], lane);
    }
    lin_cp_commit();
  };
  issue(0);
  for (int step = 0; step < nsteps; ++step) {
    if (step + 1 < nsteps) {
      issue(step + 1);
      lin_cp_wait<1>();
    } else {
      lin_cp_wait<0>();
    }
    __syncthreads();
    const int t = step / nb_, b = step - t * nb_;
    const int n0 = t * e.tnode, tn = min(e.tnode, tn_all - n0);
    const int mi = p.mul_in[b], mo = p.mul_out[b], d = p.dim[b];
    const T* xs = xbuf + (size_t)(step & 1) * e.tnode * e.rs;
    const int* nodes = s_nodes + n0;
    if (mi == 0) {
      if (!p.accumulate) {
        const int span = mo * d;
        for (int j = warp; j < tn; j += 8)
          for (int q = lane; q < span; q += 32) OUT[(size_t)nodes[j] * p.out_dim + p.out_off[b] + q] = T(0);
      }
    } else {
      const T* ws = wsm + e.w_smem_off[b];
      const int mi4 = (mi + 3) & ~3;
      const T sc = T(p.scale[b]);
      // nodes per lane: 8 warps x NB covers the tile (NB = 4 for 32-node tiles, 2 for 16-node tiles), fewer for wide irreps
#define MT_LIN_BLOCK(DD, NBB)                                                                              \
  for (int w0 = 0, lpn = lin_lpn(mo); w0 < mo; w0 += lpn)                                                  \
    for (int n0 = warp * NBB; n0 < tn; n0 += 8 * NBB)                                                      \
      lin_block<T, DD, NBB>(ws, xs + (size_t)n0 * e.rs, e.rs, mi4, mo, lpn, w0, tn - n0, nodes + n0, OUT,    \
                            p.out_dim, p.out_off[b], sc, p.accumulate)
      if (e.tnode > 16) {
        switch (d) {
          case 1: MT_LIN_BLOCK(1, 4); break;
          case 3: MT_LIN_BLOCK(3, 4); break;
          case 5: MT_LIN_BLOCK(5, 2); break;
          case 7: MT_LIN_BLOCK(7, 2); break;
          default: MT_LIN_BLOCK(9, 1); break;
        }
      } else {
        switch (d) {
          case 1: MT_LIN_BLOCK(1, 2); break;
          case 3: MT_LIN_BLOCK(3, 2); break;
          case 5: MT_LIN_BLOCK(5, 2); break;
          case 7: MT_LIN_BLOCK(7, 1); break;
          default: MT_LIN_BLOCK(9, 1); break;
        }
      }
#undef MT_LIN_BLOCK
    }
    __syncthreads();  // the buffer is refilled by step + 2
  }
}

// Warp-private variant of the same arithmetic: a warp owns NB nodes at a time and walks ALL blocks over them with
// its own double-buffered rows and its own cp.async groups -- no CTA barrier after the weight slices are in place, so
// the eight warps drift apart and one warp's copies run under another's FMAs.  (The CTA-synchronous version spent its
// time at the two barriers per block: 5.5 k of 16 k stall samples on lin2, ncu r2_lin_full.)
constexpr int kWarpNB = 2;       // nodes per warp and step
constexpr int kWarpGroupsMax = 4;  // node groups per warp: a CTA covers 8 x kWarpNB x groups nodes of one species

template <typename T>
__global__ void __launch_bounds__(256) linear_stream_kernel(const LinParams p, const LinStream e) {
  extern __shared__ __align__(16) unsigned char lin_smem[];
  __shared__ int s_nodes[8 * kWarpNB * kWarpGroupsMax];
  T* wsm = reinterpret_cast<T*>(lin_smem);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int s;
  int64_t begin, end;
  if (!lin_locate(p, e.tnode, s, begin, end)) return;  // tnode = 8 warps x kWarpNB x groups
  const int tn_all = (int)(end - begin);
  for (int i = tid; i < tn_all; i += 256) s_nodes[i] = p.sperm ? p.sperm[begin + i] : (int)(begin + i);
  const T* __restrict__ X = static_cast<const T*>(p.x);
  T* __restrict__ OUT = static_cast<T*>(p.out);
  lin_stage_weights<T>(p, e, wsm, s);
  lin_cp_commit();
  lin_cp_wait<0>();
  __syncthreads();  // weights and s_nodes in place: the only CTA-wide barrier

  // ---- from here on every warp runs on its own
  const int nb_ = p.num_blocks;
  const int ngroups = (tn_all + 8 * kWarpNB - 1) / (8 * kWarpNB);
  // my groups: node offsets (g * 8 + warp) * kWarpNB
  int mygroups = 0;
  for (int g = 0; g < ngroups; ++g)
    if ((g * 8 + warp) * kWarpNB < tn_all) ++mygroups;
  if (mygroups == 0) return;
  const int nsteps = mygroups * nb_;
  T* xw = wsm + ((e.w_total + 3) & ~3) + (size_t)warp * 2 * kWarpNB * e.rs;  // [2][kWarpNB][rs]
  auto issue = [&](int step) {
    const int g = step / nb_, b = step - g * nb_;
    const int mi = p.mul_in[b], d = p.dim[b];
    const int seg = mi * d, segp = (((mi + 3) & ~3) * d + 3) & ~3;  // copied + zero-filled up to the padded length
    const int n0 = (g * 8 + warp) * kWarpNB;
    T* buf = xw + (size_t)(step & 1) * kWarpNB * e.rs;
    if (mi > 0) {
#pragma unroll
      for (int nb = 0; nb < kWarpNB; ++nb) {
        if (n0 + nb >= tn_all) break;
        lin_stage_row<T>(buf + (size_t)nb * e.rs, X + (size_t)s_nodes[n0 + nb] * p.in_dim + p.in_off[b], seg, segp,
                         e.vec_ok[b], lane);
      }
    }
    lin_cp_commit();
  };
  issue(0);
  for (int step = 0; step < nsteps; ++step) {
    if (step + 1 < nsteps) {
      issue(step + 1);
      lin_cp_wait<1>();
    } else {
      lin_cp_wait<0>();
    }
    __syncwarp();  // every lane's copies of this step have landed
    const int g = step / nb_, b = step - g * nb_;
    const int n0 = (g * 8 + warp) * kWarpNB;
    const int ncount = min(kWarpNB, tn_all - n0);
    const int mi = p.mul_in[b], mo = p.mul_out[b], d = p.dim[b];
    const T* xs = xw + (size_t)(step & 1) * kWarpNB * e.rs;
    const int* nodes = s_nodes + n0;
    if (mi == 0) {
      if (!p.accumulate) {
        const int span = mo * d;
        for (int j = 0; j < ncount; ++j)
          for (int q = lane; q < span; q += 32) OUT[(size_t)nodes[j] * p.out_dim + p.out_off[b] + q] = T(0);
      }
    } else {
      const T* ws = wsm + e.w_smem_off[b];
      const int mi4 = (mi + 3) & ~3;
      const T sc = T(p.scale[b]);
#define MT_LIN_BLOCK(DD)                                                                                   \
  for (int w0 = 0, lpn = lin_lpn(mo); w0 < mo; w0 += lpn)                                                  \
    lin_block<T, DD, kWarpNB>(ws, xs, e.rs, mi4, mo, lpn, w0, ncount, nodes, OUT, p.out_dim, p.out_off[b], sc, \
                              p.accumulate)
      switch (d) {
        case 1: MT_LIN_BLOCK(1); break;
        case 3: MT_LIN_BLOCK(3); break;
        case 5: MT_LIN_BLOCK(5); break;
        case 7: MT_LIN_BLOCK(7); break;
        default: MT_LIN_BLOCK(9); break;
      }
#undef MT_LIN_BLOCK
    }
    __syncwarp();  // the buffer is refilled by step + 2
  }
}

// =========================================================================
// Gate (+ folded BatchNorm affine)      reference src/matten/nn/utils.py:134-140,418
// =========================================================================
template <typename T>
__global__ void __launch_bounds__(256) gate_fwd_kernel(const T* __restrict__ x, int in_dim, int out_dim,
                                                       const int32_t* __restrict__ src_idx,
                                                       const int32_t* __restrict__ gate_idx,
                                                       const int32_t* __restrict__ act_id,
                                                       const T* __restrict__ act_cst,
                                                       const T* __restrict__ aff_a,
                                                       const T* __restrict__ aff_b, T* __restrict__ out,
                                                       int64_t N) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= N * out_dim) return;
  int64_t n = t / out_dim;
  int j = (int)(t - n * out_dim);
  const T* xr = x + n * in_dim;
  T v = xr[src_idx[j]];
  int g = gate_idx[j];
  T y;
  if (g < 0) y = apply_act<T>(act_id[j], v) * act_cst[j];
  else y = v * (apply_act<T>(act_id[j], xr[g]) * act_cst[j]);
  if (aff_a) y = y * aff_a[j] + aff_b[j];
  out[t] = y;
}

// =========================================================================
// segmented pooling                     reference src/matten/nn/nodewise.py:142-148
// =========================================================================
template <typename T>
__global__ void __launch_bounds__(256) segment_reduce_kernel(const T* __restrict__ x,
                                                             const int32_t* __restrict__ ptr, int dim,
                                                             int64_t B, int mode, T* __restrict__ out) {
  int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= B * dim) return;
  int64_t b = t / dim;
  int j = (int)(t - b * dim);
  int n0 = ptr[b], n1 = ptr[b + 1];
  T acc = T(0);
  if (n1 > n0) {
    acc = x[(size_t)n0 * dim + j];
    for (int n = n0 + 1; n < n1; ++n) {
      T v = x[(size_t)n * dim + j];
      if (mode <= 1) acc += v;
      else if (mode == 2) acc = v < acc ? v : acc;
      else acc = v > acc ? v : acc;
    }
    if (mode == 1) acc = acc / T(n1 - n0);
  }
  out[t] = acc;
}

// ------------------------------------------------------------------ linear: host side
// A block, or a rectangle of one, in the orientation the kernels apply it (transposed: in and out swapped).
struct LinPiece {
  int in_off, out_off, mul_in, mul_out, dim, w_off, ld;
  double scale;
  int round;  // pieces with the same out_off before this one (linear_apply)
};

// Appends piece k as block b of a launch: its [mi4][mo] weight slice after the others, its staged rows within the
// row stride.
static void lin_layout_add(LinStream& e, int b, const LinPiece& k) {
  const int mi4 = (k.mul_in + 3) & ~3;
  e.w_smem_off[b] = e.w_total;
  e.w_total += mi4 * k.mul_out;
  e.w_total = (e.w_total + 3) & ~3;
  const int rs = ((mi4 * k.dim + 3) & ~3) + 4;
  if (rs > e.rs) e.rs = rs;
}

// dynamic shared memory of a launch that stages `rows` x rows next to its weight slices
static size_t lin_need(const LinStream& e, int rows, size_t es) {
  return ((size_t)((e.w_total + 3) & ~3) + (size_t)rows * e.rs) * es;
}

// The CTA-synchronous kernel with 8-node tiles stages 16 rows: the least shared memory of any tile, so the bound of
// what one launch can hold.
constexpr int kLinMinRows = 2 * 8;

// Cuts a piece whose weight slice and rows fit no launch into rectangles of its [mul_in x mul_out] weight that each
// fit one.  Input channels go in chunks of a multiple of 4, as large as fit.  Output channels are cut only when even
// 4 input channels of all of them do not fit: that depends on mul_out and dim alone, so the blocks that write one
// output range are cut at the same output channels and their pieces still share out_off.
static int lin_cut(const LinPiece& k, int S, int transpose, size_t es, std::vector<LinPiece>& out) {
  LinStream one;
  memset(&one, 0, sizeof(one));
  lin_layout_add(one, 0, k);
  if (lin_need(one, kLinMinRows, es) <= (size_t)kStreamSmemBytes) {
    out.push_back(k);
    return MT_OK;
  }
  const int cap = (int)(kStreamSmemBytes / es);  // elements
  // ku input channels (a multiple of 4) x kw output channels take ku * kw + kLinMinRows * (ku * dim + 4) elements
  int kw = k.mul_out;
  if (4 * kw + kLinMinRows * (4 * k.dim + 4) > cap) kw = (cap / 8) & ~3;
  const int ku = ((cap - 4 * kLinMinRows) / (kw + kLinMinRows * k.dim)) & ~3;
  for (int u0 = 0; u0 < k.mul_in; u0 += ku)
    for (int w0 = 0; w0 < k.mul_out; w0 += kw) {
      LinPiece c = k;
      c.in_off = k.in_off + u0 * k.dim;
      c.out_off = k.out_off + w0 * k.dim;
      c.mul_in = std::min(ku, k.mul_in - u0);
      c.mul_out = std::min(kw, k.mul_out - w0);
      // the weight of (u0, w0); the piece indexes from there with the whole block's row stride
      const int64_t w_off =
          k.w_off + (transpose ? (int64_t)w0 * S * k.ld + u0 : (int64_t)u0 * S * k.ld + w0);
      MT_REQUIRE(w_off < (int64_t)2147483647, "weight offset too large");
      c.w_off = (int)w_off;
      out.push_back(c);
    }
  return MT_OK;
}

// One launch of pieces pc[0..n), laid out in e: the warp-private kernel for rows of >= 512 elements when its tile
// fits, else the CTA-synchronous kernel with the largest tile that fits.
static int linear_launch(int dtype, LinParams p, LinStream e, const LinPiece* pc, int n, int accumulate,
                         cudaStream_t st) {
  const size_t es = dtype == MT_F64 ? 8 : 4;
  const int V = 16 / (int)es;
  p.num_blocks = n;
  p.accumulate = accumulate;
  for (int b = 0; b < n; ++b) {
    const LinPiece& k = pc[b];
    p.in_off[b] = k.in_off; p.out_off[b] = k.out_off; p.mul_in[b] = k.mul_in; p.mul_out[b] = k.mul_out;
    p.dim[b] = k.dim; p.w_off[b] = k.w_off; p.ld[b] = k.ld; p.scale[b] = k.scale;
    e.vec_ok[b] = (k.in_off % V == 0) && (p.in_dim % V == 0) && ((uintptr_t)p.x % 16 == 0);
    e.w_vec[b] = (k.mul_out % V == 0) && (k.ld % V == 0) && (k.w_off % V == 0) && ((uintptr_t)p.weight % 16 == 0) &&
                 k.mul_out / V <= 256;
  }
  const bool stream = p.in_dim >= 512 && lin_need(e, 8 * 2 * kWarpNB, es) <= (size_t)kStreamSmemBytes;
  size_t smem;
  if (stream) {
    // a CTA covers 8 warps x kWarpNB nodes x groups of one species; more groups amortise the weight staging, fewer
    // keep the grid above ~4 CTAs per SM
    int groups = kWarpGroupsMax;
    while (groups > 1 && p.N / (8 * kWarpNB * groups) < 4 * kNumSMs) groups >>= 1;
    e.tnode = 8 * kWarpNB * groups;
    e.tiles_per_cta = 1;
    smem = lin_need(e, 8 * 2 * kWarpNB, es);
  } else {
    // two resident CTAs per SM (16 warps, one CTA's copies under the other's arithmetic) beat one big tile
    int tnode = 32;
    while (tnode > 8 && lin_need(e, 2 * tnode, es) > (size_t)(kStreamSmemBytes / 2 - 8 * 1024)) tnode >>= 1;
    e.tnode = tnode;
    // several tiles per CTA only when that still leaves >= 4 CTAs per SM
    int tpc = (int)(p.N / ((int64_t)tnode * 4 * kNumSMs));
    e.tiles_per_cta = tpc < 1 ? 1 : (tpc > kStreamTiles ? kStreamTiles : tpc);
    smem = lin_need(e, 2 * tnode, es);
  }
  const int64_t tiles = ceil_div<int64_t>(p.N, (int64_t)e.tnode * e.tiles_per_cta) + (p.sptr ? p.S : 0);
  MT_REQUIRE(tiles < (int64_t)2147483647, "grid too large");
  MT_DISPATCH_DTYPE(dtype, {
    static thread_local bool configured = false;
    if (!configured) {
      MT_CUDA_OK(cudaFuncSetAttribute(linear_sync_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      kStreamSmemBytes));
      MT_CUDA_OK(cudaFuncSetAttribute(linear_stream_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      kStreamSmemBytes));
      configured = true;
    }
    if (stream) linear_stream_kernel<T><<<(unsigned)tiles, 256, smem, st>>>(p, e);
    else linear_sync_kernel<T><<<(unsigned)tiles, 256, smem, st>>>(p, e);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

// Applies the blocks (transposed: with in and out swapped, blocks without weights skipped) with the shapes and
// pointers of p.  Blocks that write the same output range (several input irreps of one type feeding one output,
// e3nn sums them; pieces of one cut block along its input channels) must not race: round r holds the r-th piece of
// every distinct output range, and rounds after the first accumulate.  Simplified irreps (every matten model) need
// one round.  The pieces of a round go into as few launches as fit, in order, so the result is deterministic.
static int linear_apply(int dtype, const mt_lin_block* blocks, int num_blocks, const LinParams& p, int accumulate,
                        cudaStream_t st) {
  const size_t es = dtype == MT_F64 ? 8 : 4;
  std::vector<LinPiece> pieces;  // one allocation per call; a cut block has no fixed bound on its pieces
  pieces.reserve(num_blocks);
  for (int b = 0; b < num_blocks; ++b) {
    const mt_lin_block& k = blocks[b];
    LinPiece c = {k.in_off, k.out_off, k.mul_in, k.mul_out, k.dim, k.w_off, k.mul_out, k.scale, 0};
    if (p.transpose) {
      if (k.mul_in == 0) continue;  // zero-fill blocks carry no gradient
      c.in_off = k.out_off; c.out_off = k.in_off; c.mul_in = k.mul_out; c.mul_out = k.mul_in;
    }
    int rc = lin_cut(c, p.S, p.transpose, es, pieces);
    if (rc != MT_OK) return rc;
  }
  int rounds = 0;
  for (size_t i = 0; i < pieces.size(); ++i) {
    for (size_t j = 0; j < i; ++j)
      if (pieces[j].out_off == pieces[i].out_off) ++pieces[i].round;
    if (pieces[i].round + 1 > rounds) rounds = pieces[i].round + 1;
  }
  for (int r = 0; r < rounds; ++r) {
    const int acc = (accumulate || r > 0) ? 1 : 0;
    LinPiece sel[kLinMaxBlocks];
    LinStream e;
    memset(&e, 0, sizeof(e));
    int n = 0;
    for (size_t i = 0; i < pieces.size(); ++i) {
      if (pieces[i].round != r) continue;
      LinStream grown = e;
      lin_layout_add(grown, n, pieces[i]);
      if (n > 0 && (n == kLinMaxBlocks || lin_need(grown, kLinMinRows, es) > (size_t)kStreamSmemBytes)) {
        int rc = linear_launch(dtype, p, e, sel, n, acc, st);
        if (rc != MT_OK) return rc;
        memset(&e, 0, sizeof(e));
        n = 0;
        grown = e;
        lin_layout_add(grown, n, pieces[i]);
      }
      e = grown;
      sel[n++] = pieces[i];
    }
    if (n > 0) {
      int rc = linear_launch(dtype, p, e, sel, n, acc, st);
      if (rc != MT_OK) return rc;
    }
  }
  return MT_OK;
}

int linear_check_blocks(const mt_lin_block* blocks, int num_blocks, int in_dim, int out_dim, const void* weight,
                        bool reads_weight) {
  for (int b = 0; b < num_blocks; ++b) {
    const mt_lin_block& k = blocks[b];
    // 2l+1 for l <= 4: the dims the kernels are instantiated for
    const bool dim_ok = k.dim == 1 || k.dim == 3 || k.dim == 5 || k.dim == 7 || k.dim == 9;
    MT_REQUIRE(dim_ok && k.mul_out > 0 && k.mul_in >= 0, "bad linear block %d", b);
    MT_REQUIRE(k.out_off >= 0 && k.out_off + k.mul_out * k.dim <= out_dim, "block %d exceeds out_dim", b);
    MT_REQUIRE(k.mul_in == 0 || (k.in_off >= 0 && k.in_off + k.mul_in * k.dim <= in_dim), "block %d exceeds in_dim", b);
    MT_REQUIRE(!reads_weight || k.mul_in == 0 || weight != nullptr, "null weight");
  }
  return MT_OK;
}

int linear_transposed(int dtype, const mt_lin_block* blocks, int num_blocks, int in_dim, int out_dim,
                      int num_species, const void* grad_out, const void* weight, const int32_t* species_perm,
                      const int32_t* species_ptr, int accumulate, void* grad_x, int64_t N, cudaStream_t st) {
  if (!accumulate) {
    const size_t es = dtype == MT_F64 ? 8 : 4;
    MT_CUDA_OK(cudaMemsetAsync(grad_x, 0, (size_t)N * in_dim * es, st));
  }
  LinParams p;
  memset(&p, 0, sizeof(p));
  p.in_dim = out_dim; p.out_dim = in_dim; p.S = num_species;
  p.x = grad_out; p.weight = weight; p.sperm = species_perm; p.sptr = species_ptr;
  p.transpose = 1; p.out = grad_x; p.N = N;
  return linear_apply(dtype, blocks, num_blocks, p, 1, st);
}

}  // namespace mt

using namespace mt;

extern "C" {

int mt_linear_fwd(int dtype, const mt_lin_block* blocks, int num_blocks, int in_dim, int out_dim,
                  int num_species, const void* x, const void* weight, const int32_t* species_perm,
                  const int32_t* species_ptr, int accumulate, void* out, int64_t N, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(blocks && num_blocks > 0 && num_blocks <= 4 * kLinMaxBlocks, "num_blocks %d not in 1..%d",
             num_blocks, 4 * kLinMaxBlocks);
  MT_REQUIRE(in_dim > 0 && out_dim > 0 && num_species >= 1, "bad dims");
  MT_REQUIRE((species_perm == nullptr) == (species_ptr == nullptr), "species_perm/ptr must be given together");
  MT_REQUIRE(num_species == 1 || species_ptr != nullptr, "species grouping required when num_species > 1");
  int rc = linear_check_blocks(blocks, num_blocks, in_dim, out_dim, weight, true);
  if (rc != MT_OK) return rc;
  if (N == 0) return MT_OK;
  MT_REQUIRE(x && out, "null pointer");
  LinParams p;
  memset(&p, 0, sizeof(p));
  p.in_dim = in_dim; p.out_dim = out_dim; p.S = num_species;
  p.x = x; p.weight = weight; p.sperm = species_perm; p.sptr = species_ptr;
  p.out = out; p.N = N;
  return linear_apply(dtype, blocks, num_blocks, p, accumulate, as_stream(stream));
}
int mt_gate_fwd(int dtype, const void* x, int in_dim, int out_dim, const int32_t* src_idx,
                const int32_t* gate_idx, const int32_t* act_id, const void* act_cst, const void* affine_a,
                const void* affine_b, void* out, int64_t N, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(in_dim > 0 && out_dim > 0, "bad dims");
  MT_REQUIRE((affine_a == nullptr) == (affine_b == nullptr), "affine_a/b must be given together");
  if (N == 0) return MT_OK;
  MT_REQUIRE(x && out && src_idx && gate_idx && act_id && act_cst, "null pointer");
  int64_t total = N * out_dim;
  MT_DISPATCH_DTYPE(dtype, {
    gate_fwd_kernel<T><<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, as_stream(stream)>>>(
        (const T*)x, in_dim, out_dim, src_idx, gate_idx, act_id, (const T*)act_cst, (const T*)affine_a,
        (const T*)affine_b, (T*)out, N);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

int mt_segment_reduce(int dtype, const void* x, const int32_t* ptr, int dim, int64_t B, int mode, void* out,
                      mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(dim > 0 && mode >= 0 && mode <= 3, "bad arguments");
  if (B == 0) return MT_OK;
  MT_REQUIRE(x && ptr && out, "null pointer");
  int64_t total = B * dim;
  MT_DISPATCH_DTYPE(dtype, {
    segment_reduce_kernel<T><<<(unsigned)ceil_div<int64_t>(total, 256), 256, 0, as_stream(stream)>>>(
        (const T*)x, ptr, dim, B, mode, (T*)out);
  });
  MT_LAUNCH_OK();
  return MT_OK;
}

}  // extern "C"
