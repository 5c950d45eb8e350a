// Host side of the fused convolution entry points (include/matten_b200.h: mt_conv_fwd).
#include "conv_fwd.cuh"

namespace mt {

template <typename T, int HP>
int launch_conv_fwd(const ConvFwdParams& p, int grid, int threads, size_t smem, cudaStream_t st);

#define MT_DECL(T, HP) \
  template <> int launch_conv_fwd<T, HP>(const ConvFwdParams&, int, int, size_t, cudaStream_t);
MT_DECL(float, 8) MT_DECL(float, 16) MT_DECL(float, 32) MT_DECL(float, 64)
MT_DECL(double, 8) MT_DECL(double, 16) MT_DECL(double, 32) MT_DECL(double, 64)
#undef MT_DECL

int conv_fwd_tc_try(const mt_conv_plan* plan, const void* x, const void* sh, const void* emb,
                    const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                    const int32_t* src_sorted, double avg, const void* num_neigh, void* out, void* workspace,
                    size_t workspace_bytes, const void* layout, int64_t N, int64_t E, cudaStream_t st, int* used);
size_t conv_fwd_tc_workspace_bytes(const mt_conv_plan* plan, int64_t N, int64_t E);
void conv_fwd_tc_set_debug(void* p);

// fp32 kernel of mt_conv_fwd (mt_conv_select_impl): 0 automatic, 1 tcgen05 only, 2 FMA pipes only
static int g_conv_impl = 0;

static int validate_plan(const mt_conv_plan* plan) {
  MT_REQUIRE(plan != nullptr, "null plan");
  MT_REQUIRE(plan->x_dim > 0 && plan->y_dim > 0 && plan->out_dim > 0 && plan->num_items > 0, "bad plan dims");
  MT_REQUIRE(plan->item_hdr && plan->slot_tab, "plan tables missing");
  MT_REQUIRE(plan->mlp_num_layers >= 1 && plan->mlp_num_layers <= MT_MAX_MLP_LAYERS,
             "mlp_num_layers %d not in 1..%d", plan->mlp_num_layers, MT_MAX_MLP_LAYERS);
  for (int i = 0; i <= plan->mlp_num_layers; ++i) MT_REQUIRE(plan->mlp_sizes[i] > 0, "bad mlp size");
  MT_REQUIRE(pad_hp(plan->mlp_sizes[plan->mlp_num_layers - 1]) > 0,
             "last hidden size %d > 64 not supported", plan->mlp_sizes[plan->mlp_num_layers - 1]);
  for (int i = 0; i < plan->mlp_num_layers; ++i)
    MT_REQUIRE(plan->mlp_sizes[i] <= 256, "mlp layer size %d > 256 not supported", plan->mlp_sizes[i]);
  return MT_OK;
}

template <typename T>
static int conv_fwd_impl(const mt_conv_plan* plan, const void* x, const void* sh, const void* emb,
                         const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                         const int32_t* src_sorted, double avg, const void* num_neigh, void* out, int64_t N,
                         int64_t E, cudaStream_t st) {
  ConvFwdParams p;
  memset(&p, 0, sizeof(p));
  p.x_dim = plan->x_dim;
  p.y_dim = plan->y_dim;
  p.out_dim = plan->out_dim;
  p.num_items = plan->num_items;
  p.item_hdr = plan->item_hdr;
  p.slot_tab = plan->slot_tab;
  p.nl = plan->mlp_num_layers;
  int hp_max = 8;
  for (int i = 0; i <= p.nl; ++i) p.sizes[i] = plan->mlp_sizes[i];
  for (int i = 0; i < p.nl; ++i) {
    p.w[i] = mlp_weights[i];
    int h8 = (plan->mlp_sizes[i] + 7) / 8 * 8;
    if (h8 > hp_max) hp_max = h8;
  }
  const int HP = pad_hp(p.sizes[p.nl - 1]);
  if (HP > hp_max) hp_max = HP;
  p.hp_max = hp_max;
  p.act = plan->mlp_act;
  p.act_cst = plan->mlp_act_cst;
  p.x = x; p.sh = sh; p.emb = emb;
  p.rowptr = rowptr; p.perm = perm; p.src = src_sorted;
  p.avg = avg; p.num_neigh = num_neigh; p.out = out;
  p.N = N; p.E = E;
  p.xs_stride = p.x_dim | 1;

  // chunk size from the shared-memory budget
  const size_t per_edge = (size_t)(2 * hp_max + p.xs_stride + p.y_dim) * sizeof(T);
  const size_t budget = (size_t)(sizeof(T) == 4 ? 64 : 96) * 1024;
  int EC = (int)(budget / per_edge);
  EC = EC / 8 * 8;
  if (EC > 256) EC = 256;
  if (EC < 8) EC = 8;
  p.chunk_edges = EC;
  double avg_deg = N > 0 ? (double)E / (double)N : 1.0;
  int TN = (int)((double)EC / (avg_deg > 1.0 ? avg_deg : 1.0));
  if (TN < 1) TN = 1;
  if (TN > 32) TN = 32;
  p.tile_nodes = TN;
  size_t hidden_w = 0;
  for (int i = 0; i + 1 < p.nl; ++i) hidden_w += (size_t)p.sizes[i] * p.sizes[i + 1];
  const size_t smem = (size_t)EC * per_edge + hidden_w * sizeof(T);
  MT_REQUIRE(smem <= 227 * 1024, "conv tile needs %zu bytes of shared memory", smem);
  // Resident warps per SM follow the number of contraction types the plan can touch (instruction-cache footprint: every
  // warp runs the inlined code of ONE (l1,l2,l3) type).  r1 sweep, natural irreps, 1e6 edges, fp32, ms per call with
  // (CTAs/SM x threads) = (3 x 256) / (2 x 256) / (2 x 128): sh lmax 2: 4.6 / 5.5 / 8.7; lmax 3: 16.3 / 15.2 / 25.7;
  // lmax 4: 45.0 / 36.5 / 17.0.
  const int sh_lmax = p.y_dim >= 25 ? 4 : (p.y_dim >= 16 ? 3 : 2);
  const int threads = (sizeof(T) == 4 && sh_lmax >= 4) ? 128 : 256;
  int64_t tiles = ceil_div<int64_t>(N, p.tile_nodes);
  int ctas_per_sm = (int)((227 * 1024) / (smem + 1024));
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  const int reg_limit = sizeof(T) == 4 ? (HP <= 32 ? 3 : 2) : 1;  // conv_fwd_min_blocks<T, HP>()
  if (ctas_per_sm > reg_limit) ctas_per_sm = reg_limit;
  if (sizeof(T) == 4 && sh_lmax >= 3 && ctas_per_sm > 2) ctas_per_sm = 2;
  int64_t grid = (int64_t)kNumSMs * ctas_per_sm;
  if (grid > tiles) grid = tiles;
  if (grid < 1) grid = 1;
  switch (HP) {
    case 8: return launch_conv_fwd<T, 8>(p, (int)grid, threads, smem, st);
    case 16: return launch_conv_fwd<T, 16>(p, (int)grid, threads, smem, st);
    case 32: return launch_conv_fwd<T, 32>(p, (int)grid, threads, smem, st);
    case 64: return launch_conv_fwd<T, 64>(p, (int)grid, threads, smem, st);
  }
  return set_error(MT_EINVAL, "unsupported hidden size");
}

}  // namespace mt

using namespace mt;

extern "C" {

void mt_conv_set_debug_buffer(void* device_buffer) { conv_fwd_tc_set_debug(device_buffer); }

int mt_conv_select_impl(int impl) {
  const int old = g_conv_impl;
  if (impl >= 0 && impl <= 2) g_conv_impl = impl;
  return old;
}

size_t mt_conv_fwd_workspace_bytes(const mt_conv_plan* plan, int dtype, int64_t N, int64_t E) {
  if (plan == nullptr || dtype != MT_F32 || g_conv_impl == 2) return 0;
  return conv_fwd_tc_workspace_bytes(plan, N, E);
}

int mt_conv_fwd(const mt_conv_plan* plan, int dtype, const void* x, const void* sh, const void* emb,
                const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                const int32_t* src_sorted, double avg_num_neighbors, const void* num_neigh, void* out,
                void* workspace, size_t workspace_bytes, const void* layout, int64_t N, int64_t E,
                mt_stream stream) {
  MT_ENTRY_GUARD();
  int rc = validate_plan(plan);
  if (rc != MT_OK) return rc;
  MT_REQUIRE(N >= 0 && E >= 0, "negative size");
  if (N == 0) return MT_OK;
  MT_REQUIRE(x && out && rowptr && mlp_weights, "null pointer");
  MT_REQUIRE(E == 0 || (sh && emb && perm && src_sorted), "null edge pointer");
  MT_REQUIRE(num_neigh != nullptr || avg_num_neighbors > 0.0, "avg_num_neighbors must be > 0");
  for (int i = 0; i < plan->mlp_num_layers; ++i) MT_REQUIRE(mlp_weights[i] != nullptr, "null MLP weight %d", i);
  // fp32: Blackwell tensor-core path (radial MLP on tcgen05, weights in TMEM) when the plan qualifies;
  // mt_conv_select_impl(2) forces the FMA-pipe kernel (used by the tests to cross-check the two)
  if (dtype == MT_F32) {
    const int impl = g_conv_impl;
    if (impl != 2) {
      int used = 0;
      rc = conv_fwd_tc_try(plan, x, sh, emb, mlp_weights, rowptr, perm, src_sorted, avg_num_neighbors, num_neigh,
                           out, workspace, workspace_bytes, layout, N, E, as_stream(stream), &used);
      if (rc != MT_OK) return rc;
      if (used) return MT_OK;
      if (impl == 1)
        return set_error(MT_EINVAL, "tcgen05 path requested but this plan/shape does not qualify for it");
    }
  }
  MT_DISPATCH_DTYPE(dtype, {
    return conv_fwd_impl<T>(plan, x, sh, emb, mlp_weights, rowptr, perm, src_sorted, avg_num_neighbors,
                            num_neigh, out, N, E, as_stream(stream));
  });
  return MT_OK;
}

}  // extern "C"
