// Radial MLP evaluated on its own, for MLPs too wide for the fused kernels (last hidden size in (64, 128] in the
// forward, any input / hidden size in (64, 128] in the backward): the per-edge weights w [E][Wn] are written to
// memory in receiver-sorted order, and the contractions read them from there (conv_fwd_kernel<T, 0>,
// conv_bwd_wide_kernel).
//
//   hidden layer l:  a_{l+1} = act(a_l W_l / sqrt(fan_in)) * cst        last layer:  w = a_last W_last / sqrt(H)
//
// CTA <-> a tile of kMlpEB consecutive edges.  The activations of the tile sit in shared memory, transposed
// ([k][edge], so that the 8 edges of a thread are one broadcast vector load); the current layer's weights are staged
// in k-tiles of kMlpKT rows x kMlpCW columns, pre-scaled by 1/sqrt(fan_in).  Thread (te, tc) owns edges 8 te .. 8 te + 7
// and columns tc + 32 j (j < 4) of a column chunk: 32 sums in registers, accumulated in increasing k.  Fixed order, no
// atomics: bitwise repeatable.  STORE_Z also stores the hidden pre-activations z_l [E][sizes[l+1]] for the backward.
#pragma once
#include "common.cuh"

namespace mt {

constexpr int kWideMaxH = 128;  // largest MLP input / hidden size of the wide path
constexpr int kMlpEB = 64;      // edges per CTA tile
constexpr int kMlpAS = kMlpEB + 4;  // row stride of the transposed activation tiles (16-byte aligned rows)
constexpr int kMlpCW = 128;     // weight columns per chunk
constexpr int kMlpKT = 32;      // weight rows per staged k-tile

struct RadialMlpParams {
  int nl;
  int sizes[MT_MAX_MLP_LAYERS + 1];
  int act;
  double act_cst;
  const void* w[MT_MAX_MLP_LAYERS];
  const void* emb;             // [E][sizes[0]] in the caller's edge order, read through perm
  const int32_t* perm;
  int64_t E;
  int rows;                    // rows of the activation tiles: largest input / hidden size
  void* out;                   // [E][sizes[nl]] per-edge weights, receiver-sorted order
  void* z[MT_MAX_MLP_LAYERS];  // STORE_Z: z[l] [E][sizes[l+1]] for l < nl - 1
};

template <typename T>
__device__ __forceinline__ void mlp_load4(const T* p, T (&v)[4]);
template <>
__device__ __forceinline__ void mlp_load4<float>(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void mlp_load4<double>(const double* p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

template <typename T, bool STORE_Z>
__global__ void __launch_bounds__(256, 1) radial_mlp_kernel(const RadialMlpParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* buf0 = reinterpret_cast<T*>(smem_raw);  // [rows][kMlpAS]
  T* buf1 = buf0 + (size_t)p.rows * kMlpAS;  // [rows][kMlpAS]
  T* Ws = buf1 + (size_t)p.rows * kMlpAS;    // [kMlpKT][kMlpCW]
  const int tid = threadIdx.x, te = tid >> 5, tc = tid & 31;
  const int in0 = p.sizes[0];
  const T cst = T(p.act_cst);
  const T* __restrict__ EMB = static_cast<const T*>(p.emb);
  using P = typename pair_of<T>::type;  // edge pairs: one FFMA2 (broadcast weight) per pair in fp32
  const int64_t nchunks = ceil_div<int64_t>(p.E, kMlpEB);
  for (int64_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const int64_t e0 = ch * kMlpEB;
    const int ne = (int)imin64(kMlpEB, p.E - e0);
    __syncthreads();  // the previous tile's activations have been consumed
    for (int t = tid; t < in0 * kMlpEB; t += blockDim.x) {
      const int k = t / kMlpEB, el = t - k * kMlpEB;
      buf0[k * kMlpAS + el] = el < ne ? EMB[(size_t)p.perm[e0 + el] * in0 + k] : T(0);
    }
    T* hin = buf0;
    T* hout = buf1;
    for (int l = 0; l < p.nl; ++l) {
      const int fi = p.sizes[l], fo = p.sizes[l + 1];
      const bool last = l + 1 == p.nl;
      const T s = T(1) / sqrt(T(fi));
      const T* __restrict__ Wg = static_cast<const T*>(p.w[l]);
      for (int cb = 0; cb < fo; cb += kMlpCW) {
        P acc[4][4];  // [column j][edge pair i]
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[j][i].x = acc[j][i].y = T(0);
        for (int kb = 0; kb < fi; kb += kMlpKT) {
          const int kn = min(kMlpKT, fi - kb);
          __syncthreads();  // Ws is free, hin is complete
          for (int t = tid; t < kMlpKT * kMlpCW; t += blockDim.x) {
            const int kk = t / kMlpCW, c = t - kk * kMlpCW;
            Ws[t] = (kk < kn && cb + c < fo) ? Wg[(size_t)(kb + kk) * fo + cb + c] * s : T(0);
          }
          __syncthreads();
          for (int kk = 0; kk < kn; ++kk) {
            T h0[4], h1[4];  // edges 8 te .. 8 te + 3, 8 te + 4 .. 8 te + 7
            const T* hr = hin + (size_t)(kb + kk) * kMlpAS + te * 8;
            mlp_load4<T>(hr, h0);
            mlp_load4<T>(hr + 4, h1);
            const T* wr = Ws + kk * kMlpCW + tc;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const T wv = wr[32 * j];
              fma_pair(wv, h0[0], h0[1], acc[j][0]);
              fma_pair(wv, h0[2], h0[3], acc[j][1]);
              fma_pair(wv, h1[0], h1[1], acc[j][2]);
              fma_pair(wv, h1[2], h1[3], acc[j][3]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = cb + tc + 32 * j;
          if (c >= fo) continue;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int el = te * 8 + i;
            const T v = (i & 1) ? acc[j][i >> 1].y : acc[j][i >> 1].x;
            if (last) {
              if (el < ne) static_cast<T*>(p.out)[(size_t)(e0 + el) * fo + c] = v;
            } else {
              if constexpr (STORE_Z)
                if (el < ne) static_cast<T*>(p.z[l])[(size_t)(e0 + el) * fo + c] = v;
              hout[(size_t)c * kMlpAS + el] = apply_act<T>(p.act, v) * cst;
            }
          }
        }
      }
      T* tmp = hin; hin = hout; hout = tmp;
    }
  }
}

// one launch over all E edges; the caller has checked every input / hidden size <= kWideMaxH
template <typename T, bool STORE_Z>
inline int launch_radial_mlp(const RadialMlpParams& p, cudaStream_t st) {
  if (p.E == 0) return MT_OK;
  const size_t smem = ((size_t)2 * p.rows * kMlpAS + (size_t)kMlpKT * kMlpCW) * sizeof(T);
  static thread_local size_t configured = 0;
  if (smem > configured) {
    MT_CUDA_OK(cudaFuncSetAttribute(radial_mlp_kernel<T, STORE_Z>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    configured = smem;
  }
  const int per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));
  const int64_t chunks = ceil_div<int64_t>(p.E, kMlpEB);
  int64_t grid = (int64_t)kNumSMs * (per_sm > 1 ? per_sm : 1);
  if (grid > chunks) grid = chunks;
  radial_mlp_kernel<T, STORE_Z><<<(unsigned)grid, 256, smem, st>>>(p);
  MT_LAUNCH_OK();
  return MT_OK;
}

// rows of the activation tiles: the largest layer input
inline int radial_mlp_rows(const mt_conv_plan* plan) {
  int r = 1;
  for (int i = 0; i < plan->mlp_num_layers; ++i) r = plan->mlp_sizes[i] > r ? plan->mlp_sizes[i] : r;
  return r;
}

// per-edge weight buffer of the wide path: E x Wn values
inline size_t radial_mlp_out_bytes(const mt_conv_plan* plan, size_t es, int64_t E) {
  return align256((size_t)E * plan->mlp_sizes[plan->mlp_num_layers] * es);
}

}  // namespace mt
