// Host side of mt_conv_bwd / mt_conv_bwd_full (include/matten_b200.h): workspace carve-up and the K0..K4 launches.
#include "conv_bwd.cuh"

namespace mt {

struct BwdLayout {
  size_t z_off[MT_MAX_MLP_LAYERS];
  size_t dw_off, dxe_off, dhp_off, partl_off, parth_off, total;
  int ncg, grid2, grid3, hid_numel, hid_eb, rs;
  bool wide;                 // an input / hidden size above kBwdMaxH: the wide kernels
  size_t wpe_off, da_off[2];  // wide: per-edge weights [E][Wn]; da of the hidden layers [E][<= 128], ping-pong
};

static bool wide_bwd(const mt_conv_plan* plan) {
  for (int i = 0; i < plan->mlp_num_layers; ++i)
    if (plan->mlp_sizes[i] > kBwdMaxH) return true;
  return false;
}

static BwdLayout bwd_layout(const mt_conv_plan* plan, size_t es, int64_t E) {
  BwdLayout L;
  memset(&L, 0, sizeof(L));
  const int nl = plan->mlp_num_layers;
  const int H = plan->mlp_sizes[nl - 1], Wn = plan->mlp_sizes[nl];
  size_t o = 0;
  int hid = 0;
  for (int l = 0; l + 1 < nl; ++l) {
    L.z_off[l] = o;
    o += align256((size_t)E * plan->mlp_sizes[l + 1] * es);
    hid += plan->mlp_sizes[l] * plan->mlp_sizes[l + 1];
  }
  L.hid_numel = hid;
  L.wide = wide_bwd(plan);
  L.ncg = ceil_div<int>(Wn, kLastCW);
  const int64_t chunks2 = ceil_div<int64_t>(E, L.wide && H > kBwdMaxH ? kLastEBWide : kLastEB);
  L.grid2 = (int)(chunks2 < 2 * kNumSMs ? (chunks2 > 0 ? chunks2 : 1) : 2 * kNumSMs);
  int hmax = 1;
  for (int i = 0; i < nl; ++i) hmax = plan->mlp_sizes[i] > hmax ? plan->mlp_sizes[i] : hmax;
  L.rs = hmax + 1;
  L.hid_eb = kHidEBMax;
  while (L.hid_eb > 16 && ((size_t)3 * L.hid_eb * L.rs + (size_t)L.rs * L.rs + hid) * es > 36 * 1024) L.hid_eb >>= 1;
  const int64_t chunks3 = ceil_div<int64_t>(E, L.hid_eb);
  L.grid3 = (int)(chunks3 < 6 * kNumSMs ? (chunks3 > 0 ? chunks3 : 1) : 6 * kNumSMs);  // small tiles: 6 CTAs per SM
  if (L.wide) {  // one CTA per SM in fp64 (W_l of 128 x 129 plus the tiles: ~200 KB), two in fp32
    const int64_t chunks3w = ceil_div<int64_t>(E, kHidWideEB);
    const int64_t cap = (int64_t)kNumSMs * (es == 4 ? 2 : 1);
    L.grid3 = (int)(chunks3w < cap ? (chunks3w > 0 ? chunks3w : 1) : cap);
  }
  L.dw_off = o;
  o += align256((size_t)E * Wn * es);
  L.dxe_off = o;
  o += align256((size_t)E * plan->x_dim * es);
  L.dhp_off = o;
  o += align256((size_t)L.ncg * E * H * es);
  L.partl_off = o;
  o += align256((size_t)L.grid2 * H * Wn * es);
  L.parth_off = o;
  {  // one partial per CTA of the generic K3, one per warp of the fast K3
    const size_t rows = (size_t)L.grid3 > (size_t)kHidFastCtas * kHidFastWarps ? (size_t)L.grid3
                                                                               : (size_t)kHidFastCtas * kHidFastWarps;
    o += align256(rows * (hid > 0 ? hid : 1) * es);
  }
  if (L.wide) {
    L.wpe_off = o;
    o += radial_mlp_out_bytes(plan, es, E);
    for (int i = 0; i < 2 && nl > 2; ++i) {
      L.da_off[i] = o;
      o += align256((size_t)E * hmax * es);
    }
  }
  L.total = o;
  return L;
}

template <typename T, int HP>
static int launch_last(const ConvBwdParams& p, cudaStream_t st) {
  const size_t smem = ((size_t)kLastEB * (kLastCW + 4) + (size_t)kLastEB * HP + (size_t)kLastCW * HP) * sizeof(T);
  MT_CUDA_OK(cudaFuncSetAttribute(mlp_bwd_last_kernel<T, HP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(p.grid2, p.ncg);
  mlp_bwd_last_kernel<T, HP><<<grid, 256, smem, st>>>(p);
  MT_LAUNCH_OK();
  return MT_OK;
}

template <typename T>
static int launch_last_wide(const ConvBwdParams& p, cudaStream_t st) {
  const size_t smem = ((size_t)kLastEBWide * (kLastCW + 4) + (size_t)kLastEBWide * kWideMaxH +
                       (size_t)kLastCW * kWideMaxH) * sizeof(T);
  MT_CUDA_OK(cudaFuncSetAttribute(mlp_bwd_last_wide_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(p.grid2, p.ncg);
  mlp_bwd_last_wide_kernel<T><<<grid, 256, smem, st>>>(p);
  MT_LAUNCH_OK();
  return MT_OK;
}

// wide K3: one launch per hidden layer, from the last down, then the fixed-order sums of the per-CTA partials
template <typename T>
static int launch_hidden_wide(const ConvBwdParams& p, const BwdLayout& L, unsigned char* ws, void* const* grad_w,
                              bool emb, cudaStream_t st) {
  int woff = p.hid_numel;
  const T* da_in = static_cast<const T*>(p.DHP);
  int parts = p.ncg;
  for (int l = p.nl - 2; l >= 0; --l) {
    const int fi = p.sizes[l], fo = p.sizes[l + 1];
    woff -= fi * fo;
    T* da_out = l > 0 ? reinterpret_cast<T*>(ws + L.da_off[l & 1]) : nullptr;
    const size_t smem = ((size_t)2 * kHidWideEB * kHidWideRS + (size_t)fi * (fo + 1)) * sizeof(T);
    if (l == 0 && emb) {
      MT_CUDA_OK(cudaFuncSetAttribute(mlp_bwd_hidden_wide_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
      mlp_bwd_hidden_wide_kernel<T, true><<<p.grid3, 256, smem, st>>>(p, l, da_in, parts, da_out, woff);
    } else {
      MT_CUDA_OK(cudaFuncSetAttribute(mlp_bwd_hidden_wide_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
      mlp_bwd_hidden_wide_kernel<T, false><<<p.grid3, 256, smem, st>>>(p, l, da_in, parts, da_out, woff);
    }
    MT_LAUNCH_OK();
    da_in = da_out;
    parts = 1;
  }
  int64_t off = 0;
  for (int l = 0; grad_w && l + 1 < p.nl; ++l) {
    const int64_t cnt = (int64_t)p.sizes[l] * p.sizes[l + 1];
    reduce_partials_kernel<T><<<(unsigned)ceil_div<int64_t>(cnt, 32), 256, 0, st>>>(
        static_cast<const T*>(p.PARTH), p.hid_numel, p.grid3, off, cnt, T(1) / sqrt(T(p.sizes[l])),
        static_cast<T*>(grad_w[l]));
    MT_LAUNCH_OK();
    off += cnt;
  }
  return MT_OK;
}

// K1: tile geometry from the shared-memory budget (two CTAs per SM when possible)
template <typename T, bool EG, bool WIDE>
static int launch_conv_bwd_k1(ConvBwdParams& p, int64_t N, int64_t E, cudaStream_t st) {
  const double avg_deg = N > 0 ? (double)E / (double)N : 1.0;
  const size_t fixed = (size_t)p.num_paths * 16;
  // resident CTAs per SM the register budget allows (launch bounds of conv_bwd_kernel) -> shared-memory budget per CTA:
  // the kernel alternates staging / GEMM / contraction phases between barriers, so more small CTAs hide more of it
  const int threads1 = 128;  // more, smaller CTAs hide the phase barriers better (r1 sweep)
  const int per_sm_regs = (sizeof(T) == 4 ? 3 : 2) * (256 / threads1) - (WIDE ? 256 / threads1 : 0);
  const size_t budget = (size_t)(227 * 1024) / per_sm_regs - 1024;
  // EG: one sh-gradient partial row per (item, staged edge)
  const size_t per_edge_eg = EG ? (size_t)p.num_items * p.y_dim : 0;
  int EC = 32, TN = 1;
  size_t smem = 0;
  for (;;) {
    TN = (int)((double)EC / (avg_deg > 1.0 ? avg_deg : 1.0));
    if (TN < 1) TN = 1;
    if (TN > 16) TN = 16;
    for (;;) {
      smem = fixed + ((size_t)EC * (p.hs_stride + p.xs_stride + p.y_dim + p.wt_stride + per_edge_eg) + (size_t)TN * (p.out_dim + 1)) * sizeof(T) +
             (size_t)EC * sizeof(int);
      if (smem <= budget || TN == 1) break;
      TN = TN / 2;
    }
    if (smem <= budget || EC == 8) break;
    EC /= 2;
  }
  MT_REQUIRE(smem <= 227 * 1024, "conv_bwd tile needs %zu bytes of shared memory", smem);
  p.chunk_edges = EC;
  p.tile_nodes = TN;
  static thread_local size_t cfg1 = 0;
  const auto kernel = WIDE ? conv_bwd_wide_kernel<T, EG> : conv_bwd_kernel<T, EG>;
  if (smem > cfg1) {
    MT_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cfg1 = smem;
  }
  const int64_t tiles = ceil_div<int64_t>(N, TN);
  int per_sm = (int)((size_t)(227 * 1024) / (smem + 1024));
  if (per_sm > per_sm_regs) per_sm = per_sm_regs;
  if (per_sm < 1) per_sm = 1;
  int64_t grid = (int64_t)kNumSMs * per_sm;
  if (grid > tiles) grid = tiles;
  kernel<<<(int)grid, threads1, smem, st>>>(p);
  MT_LAUNCH_OK();
  return MT_OK;
}

template <typename T>
static int conv_bwd_impl(const mt_conv_plan* plan, const void* x, const void* sh, const void* emb,
                         const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                         const int32_t* src_sorted, const int32_t* sender_ptr, const int32_t* sender_perm, double avg,
                         const void* num_neigh, const void* grad_out, void* grad_x, void* const* grad_w,
                         void* grad_sh, void* grad_emb, void* workspace, size_t workspace_bytes, int64_t N, int64_t E,
                         cudaStream_t st, int dtype) {
  const int nl = plan->mlp_num_layers;
  const int H = plan->mlp_sizes[nl - 1], Wn = plan->mlp_sizes[nl];
  if (E == 0) {  // no edges: all gradients are zero
    if (grad_x) MT_CUDA_OK(cudaMemsetAsync(grad_x, 0, (size_t)N * plan->x_dim * sizeof(T), st));
    if (grad_w)
      for (int l = 0; l < nl; ++l)
        MT_CUDA_OK(cudaMemsetAsync(grad_w[l], 0, (size_t)plan->mlp_sizes[l] * plan->mlp_sizes[l + 1] * sizeof(T), st));
    return MT_OK;
  }
  const BwdLayout L = bwd_layout(plan, sizeof(T), E);
  MT_REQUIRE(workspace != nullptr && workspace_bytes >= L.total, "conv_bwd workspace too small: %zu < %zu",
             workspace_bytes, L.total);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  ConvBwdParams p;
  memset(&p, 0, sizeof(p));
  p.x_dim = plan->x_dim; p.y_dim = plan->y_dim; p.out_dim = plan->out_dim; p.Wn = Wn;
  p.num_items = plan->bw_num_items; p.num_paths = plan->bw_num_paths;
  p.item_hdr = plan->bw_item_hdr; p.lane_tab = plan->bw_lane_tab; p.path_tab = plan->bw_path_tab;
  p.nl = nl;
  for (int i = 0; i <= nl; ++i) p.sizes[i] = plan->mlp_sizes[i];
  p.act = plan->mlp_act; p.act_cst = plan->mlp_act_cst;
  for (int l = 0; l < nl; ++l) p.w[l] = mlp_weights[l];
  for (int l = 0; l + 1 < nl; ++l) p.z[l] = ws + L.z_off[l];
  p.x = x; p.sh = sh; p.emb = emb; p.rowptr = rowptr; p.perm = perm; p.src = src_sorted;
  p.avg = avg; p.num_neigh = num_neigh; p.g = grad_out;
  p.DW = ws + L.dw_off; p.DXE = ws + L.dxe_off; p.DHP = ws + L.dhp_off;
  p.PARTL = ws + L.partl_off; p.PARTH = ws + L.parth_off;
  p.N = N; p.E = E;
  p.ncg = L.ncg; p.grid2 = L.grid2; p.grid3 = L.grid3; p.hid_numel = L.hid_numel;
  p.xs_stride = p.x_dim | 1;
  p.hs_stride = L.wide ? 0 : (H + 3) / 4 * 4;  // the wide K1 stages no last-layer input
  p.wt_stride = Wn;
  p.rs = L.rs;
  p.hid_eb = L.hid_eb;
  p.gsh = grad_sh;
  p.gemb = grad_emb;
  if (L.wide) p.wpe = ws + L.wpe_off;

  // the MLP shape of the matten configs in fp32 takes the lane-per-edge kernels
  const bool fast_mlp = sizeof(T) == 4 && nl == 3 && p.sizes[0] <= 8 && p.sizes[1] == 32 && p.sizes[2] == 32 &&
                        p.act == MT_ACT_SILU;
  // K0: hidden pre-activations (wide: and the per-edge weights)
  if (L.wide) {
    RadialMlpParams m;
    memset(&m, 0, sizeof(m));
    m.nl = nl;
    for (int i = 0; i <= nl; ++i) m.sizes[i] = p.sizes[i];
    for (int i = 0; i < nl; ++i) m.w[i] = p.w[i];
    for (int i = 0; i + 1 < nl; ++i) m.z[i] = p.z[i];
    m.act = p.act; m.act_cst = p.act_cst;
    m.emb = emb; m.perm = perm; m.E = E;
    m.rows = radial_mlp_rows(plan);
    m.out = ws + L.wpe_off;
    const int rc = launch_radial_mlp<T, true>(m, st);
    if (rc != MT_OK) return rc;
  } else if (fast_mlp) {
    int64_t g0 = ceil_div<int64_t>(E, 256);
    if (g0 > (int64_t)kNumSMs * 8) g0 = (int64_t)kNumSMs * 8;
    edge_hidden_fast_kernel<<<(unsigned)g0, 256, 0, st>>>(p);
    MT_LAUNCH_OK();
  } else if (nl > 1) {
    const size_t smem0 = ((size_t)p.hid_eb * p.rs + (size_t)p.rs * p.rs) * sizeof(T);
    static thread_local size_t cfg0 = 0;
    if (smem0 > cfg0) {
      MT_CUDA_OK(cudaFuncSetAttribute(edge_hidden_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0));
      cfg0 = smem0;
    }
    const int64_t chunks = ceil_div<int64_t>(E, p.hid_eb);
    const int grid0 = (int)(chunks < 12 * kNumSMs ? chunks : 12 * kNumSMs);
    edge_hidden_kernel<T><<<grid0, 256, smem0, st>>>(p);
    MT_LAUNCH_OK();
  }
  {
    const int rc = L.wide ? (grad_sh ? launch_conv_bwd_k1<T, true, true>(p, N, E, st)
                                     : launch_conv_bwd_k1<T, false, true>(p, N, E, st))
                          : (grad_sh ? launch_conv_bwd_k1<T, true, false>(p, N, E, st)
                                     : launch_conv_bwd_k1<T, false, false>(p, N, E, st));
    if (rc != MT_OK) return rc;
  }
  // per-sender sum of the per-edge input gradients
  if (grad_x) {
    int rc = mt_segment_sum_gather(dtype, p.DXE, sender_perm, sender_ptr, p.x_dim, N, E, grad_x, st);
    if (rc != MT_OK) return rc;
  }
  // K2 / K3 give the weight gradients and, through da of the first layer, the embedding gradient
  if (grad_w || grad_emb) {
    int rc = MT_OK;
    if (H > kBwdMaxH) rc = launch_last_wide<T>(p, st);
    else switch (pad_hp(H)) {
      case 8: rc = launch_last<T, 8>(p, st); break;
      case 16: rc = launch_last<T, 16>(p, st); break;
      case 32: rc = launch_last<T, 32>(p, st); break;
      default: rc = launch_last<T, 64>(p, st); break;
    }
    if (rc != MT_OK) return rc;
    if (grad_w) {
      const int64_t cnt = (int64_t)H * Wn;
      reduce_partials_kernel<T><<<(unsigned)ceil_div<int64_t>(cnt, 32), 256, 0, st>>>(
          static_cast<const T*>(p.PARTL), cnt, p.grid2, 0, cnt, T(1) / sqrt(T(H)), static_cast<T*>(grad_w[nl - 1]));
      MT_LAUNCH_OK();
    }
    if (nl == 1) {
      if (grad_emb) {
        int64_t ge = ceil_div<int64_t>(E * H, 256);
        if (ge > (int64_t)kNumSMs * 8) ge = (int64_t)kNumSMs * 8;
        emb_grad_last_kernel<T><<<(unsigned)ge, 256, 0, st>>>(p);
        MT_LAUNCH_OK();
      }
    } else if (L.wide) {
      rc = launch_hidden_wide<T>(p, L, ws, grad_w, grad_emb != nullptr, st);
      if (rc != MT_OK) return rc;
    } else if (fast_mlp) {
      int64_t gf = ceil_div<int64_t>(ceil_div<int64_t>(E, 32), kHidFastWarps);
      if (gf > kHidFastCtas) gf = kHidFastCtas;
      if (grad_emb) mlp_bwd_hidden_fast_kernel<true><<<(unsigned)gf, 32 * kHidFastWarps, 0, st>>>(p);
      else mlp_bwd_hidden_fast_kernel<false><<<(unsigned)gf, 32 * kHidFastWarps, 0, st>>>(p);
      MT_LAUNCH_OK();
      const int nparts = (int)gf * kHidFastWarps;
      int64_t off = 0;
      for (int l = 0; grad_w && l + 1 < nl; ++l) {
        const int64_t cnt = (int64_t)p.sizes[l] * p.sizes[l + 1];
        reduce_partials_kernel<T><<<(unsigned)ceil_div<int64_t>(cnt, 32), 256, 0, st>>>(
            static_cast<const T*>(p.PARTH), p.hid_numel, nparts, off, cnt, T(1) / sqrt(T(p.sizes[l])),
            static_cast<T*>(grad_w[l]));
        MT_LAUNCH_OK();
        off += cnt;
      }
    } else {
      const size_t smem3 = ((size_t)3 * p.hid_eb * p.rs + (size_t)p.rs * p.rs + p.hid_numel) * sizeof(T);
      MT_REQUIRE(smem3 <= 227 * 1024, "hidden MLP too large for the backward kernel");
      if (grad_emb) {
        static thread_local size_t cfg3e = 0;
        if (smem3 > cfg3e) {
          MT_CUDA_OK(cudaFuncSetAttribute(mlp_bwd_hidden_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem3));
          cfg3e = smem3;
        }
        mlp_bwd_hidden_kernel<T, true><<<p.grid3, 256, smem3, st>>>(p);
      } else {
        static thread_local size_t cfg3 = 0;
        if (smem3 > cfg3) {
          MT_CUDA_OK(cudaFuncSetAttribute(mlp_bwd_hidden_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem3));
          cfg3 = smem3;
        }
        mlp_bwd_hidden_kernel<T, false><<<p.grid3, 256, smem3, st>>>(p);
      }
      MT_LAUNCH_OK();
      int64_t off = 0;
      for (int l = 0; grad_w && l + 1 < nl; ++l) {
        const int64_t cnt = (int64_t)p.sizes[l] * p.sizes[l + 1];
        reduce_partials_kernel<T><<<(unsigned)ceil_div<int64_t>(cnt, 32), 256, 0, st>>>(
            static_cast<const T*>(p.PARTH), p.hid_numel, p.grid3, off, cnt, T(1) / sqrt(T(p.sizes[l])),
            static_cast<T*>(grad_w[l]));
        MT_LAUNCH_OK();
        off += cnt;
      }
    }
  }
  return MT_OK;
}

}  // namespace mt

using namespace mt;

extern "C" {

size_t mt_conv_bwd_workspace_bytes(const mt_conv_plan* plan, int dtype, int64_t N, int64_t E) {
  (void)N;
  if (plan == nullptr || E <= 0 || plan->mlp_num_layers < 1 || plan->mlp_num_layers > MT_MAX_MLP_LAYERS) return 0;
  return bwd_layout(plan, dtype == MT_F64 ? 8 : 4, E).total;
}

int mt_conv_bwd_full(const mt_conv_plan* plan, int dtype, const void* x, const void* sh, const void* emb,
                     const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                     const int32_t* src_sorted, const int32_t* sender_ptr, const int32_t* sender_perm,
                     double avg_num_neighbors, const void* num_neigh, const void* grad_out, void* grad_x,
                     void* const* grad_mlp_weights, void* grad_sh, void* grad_emb, void* workspace,
                     size_t workspace_bytes, int64_t N, int64_t E, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(plan != nullptr, "null plan");
  MT_REQUIRE(plan->bw_num_items > 0 && plan->bw_item_hdr && plan->bw_lane_tab && plan->bw_path_tab,
             "plan has no backward tables");
  MT_REQUIRE(plan->mlp_num_layers >= 1 && plan->mlp_num_layers <= MT_MAX_MLP_LAYERS, "bad mlp_num_layers");
  for (int i = 0; i < plan->mlp_num_layers; ++i)
    MT_REQUIRE(plan->mlp_sizes[i] > 0 && plan->mlp_sizes[i] <= kWideMaxH,
               "conv_bwd supports MLP input/hidden sizes <= %d, got %d", kWideMaxH, plan->mlp_sizes[i]);
  MT_REQUIRE(N >= 0 && E >= 0, "negative size");
  if (N == 0) return MT_OK;
  MT_REQUIRE(x && rowptr && mlp_weights && grad_out, "null pointer");
  MT_REQUIRE(E == 0 || (sh && emb && perm && src_sorted), "null edge pointer");
  MT_REQUIRE(grad_x == nullptr || E == 0 || (sender_ptr && sender_perm), "sender CSR required for grad_x");
  MT_REQUIRE(num_neigh != nullptr || avg_num_neighbors > 0.0, "avg_num_neighbors must be > 0");
  for (int i = 0; i < plan->mlp_num_layers; ++i) {
    MT_REQUIRE(mlp_weights[i] != nullptr, "null MLP weight %d", i);
    MT_REQUIRE(grad_mlp_weights == nullptr || grad_mlp_weights[i] != nullptr, "null MLP weight gradient %d", i);
  }
  MT_DISPATCH_DTYPE(dtype, {
    return conv_bwd_impl<T>(plan, x, sh, emb, mlp_weights, rowptr, perm, src_sorted, sender_ptr, sender_perm,
                            avg_num_neighbors, num_neigh, grad_out, grad_x, grad_mlp_weights, grad_sh, grad_emb,
                            workspace, workspace_bytes, N, E, as_stream(stream), dtype);
  });
  return MT_OK;
}

int mt_conv_bwd(const mt_conv_plan* plan, int dtype, const void* x, const void* sh, const void* emb,
                const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                const int32_t* src_sorted, const int32_t* sender_ptr, const int32_t* sender_perm,
                double avg_num_neighbors, const void* num_neigh, const void* grad_out, void* grad_x,
                void* const* grad_mlp_weights, void* workspace, size_t workspace_bytes, int64_t N, int64_t E,
                mt_stream stream) {
  return mt_conv_bwd_full(plan, dtype, x, sh, emb, mlp_weights, rowptr, perm, src_sorted, sender_ptr, sender_perm,
                          avg_num_neighbors, num_neigh, grad_out, grad_x, grad_mlp_weights, nullptr, nullptr,
                          workspace, workspace_bytes, N, E, stream);
}

}  // extern "C"
