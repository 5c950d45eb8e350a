// Host launcher of the tcgen05 convolution forward (see conv_fwd_tc.cuh).
#include <stdlib.h>

#include <cub/device/device_scan.cuh>

#include "conv_fwd_tc.cuh"

namespace mt {

constexpr size_t kTcSmemLimit = (size_t)227 * 1024 - 1024;  // dynamic + static shared memory must fit 227 KB

// widest chunk (MMA N, a multiple of 16) whose staging buffers fit the shared memory; 0: none
static int tc_pick_ne(const mt_conv_tc_part& part, int y_lmax) {
  static const int cand[] = {256, 128, 80, 64, 48, 32};
  const int y_pad = sh_pad_len(y_lmax);
  for (int ne : cand) {
    if (2 * part.num_tiles * ne > 512) continue;
    const TcSmemLayout L = tc_smem_layout(part.a_rows, part.x_cols, y_pad, part.num_bi, ne);
    if (L.total <= kTcSmemLimit) return ne;
  }
  return 0;
}

static bool tc_plan_qualifies(const mt_conv_plan* plan) {
  if (plan->tc_num_parts <= 0 || plan->tc_num_parts > MT_TC_MAX_PARTS) return false;
  if (plan->tc_y_lmax < 0 || plan->tc_y_lmax > MT_LMAX) return false;
  if (plan->mlp_num_layers > 3) return false;  // at most two hidden layers are kept in registers
  for (int i = 0; i < plan->mlp_num_layers; ++i)
    if (plan->mlp_sizes[i] > kTcK) return false;
  if ((plan->x_dim & 3) != 0) return false;  // TMA: rows must be multiples of 16 bytes
  for (int i = 0; i < plan->tc_num_parts; ++i) {
    const mt_conv_tc_part& pt = plan->tc_parts[i];
    if (pt.num_tiles <= 0 || pt.num_tiles > kTcMaxTiles || pt.num_bi <= 0 || pt.num_bi > kTcMaxBI) return false;
    if (pt.a_rows <= 0 || pt.a_rows > pt.num_tiles * 128 || (pt.a_rows & 31) != 0) return false;
    if (!pt.row_wcol || !pt.bi_hdr || !pt.bi_lane || !pt.q_list) return false;
    if (pt.x_cols <= 0 || pt.x_cols > 256 || (pt.x_cols & 7) != 0 || (pt.x_lo & 3) != 0) return false;
    if (tc_pick_ne(pt, plan->tc_y_lmax) == 0) return false;
  }
  return true;
}

// The per-batch edge layout: the padded column order of the receiver-sorted edge list and the pair-interleaved sh rows
// the fused kernel streams per column.  mt_conv_layout_prepare builds it once per batch in the caller's buffer; a call
// without a layout builds it at the start of its own workspace.
struct TcLayout {
  size_t rowptr_pad, scan_tmp, orig_pad, src_pad, ypairs, total;
  int64_t cols_max;
  size_t scan_bytes;
};
static TcLayout tc_layout(int y_lmax, int64_t N, int64_t E) {
  TcLayout w;
  w.cols_max = (E + 3 * N + 3) & ~(int64_t)3;
  if (w.cols_max < 4) w.cols_max = 4;
  w.scan_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, w.scan_bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (int)(N + 1));
  size_t o = 0;
  w.rowptr_pad = o;
  o += align256((size_t)(N + 1) * 4 * 2);  // padded degrees, then their scan
  w.scan_tmp = o;
  o += align256(w.scan_bytes);
  w.orig_pad = o;
  o += align256((size_t)w.cols_max * 4);
  w.src_pad = o;
  o += align256((size_t)w.cols_max * 4);
  w.ypairs = o;
  o += align256((size_t)(w.cols_max / 2) * 2 * sh_pad_len(y_lmax) * 4);
  w.total = o;
  return w;
}

// workspace of a call: the layout, the h planes of the layer (192 bytes per column) and slack to align the buffer to
// 256 bytes
static size_t tc_workspace_bytes(const TcLayout& L) { return L.total + align256((size_t)L.cols_max * 192) + 256; }

// fills the layout L at `base` (256-byte aligned): padded column order, then the sh pair rows
static int tc_prepare_layout(const TcLayout& L, uintptr_t base, int y_lmax, const float* sh, const int32_t* rowptr,
                             const int32_t* perm, const int32_t* src_sorted, int64_t N, cudaStream_t st) {
  int32_t* degp = reinterpret_cast<int32_t*>(base + L.rowptr_pad);
  int32_t* rowptr_pad = degp + (N + 1);
  int32_t* orig_pad = reinterpret_cast<int32_t*>(base + L.orig_pad);
  tc_pad_degree_kernel<<<(unsigned)ceil_div<int64_t>(N + 1, 256), 256, 0, st>>>(rowptr, N, degp);
  MT_LAUNCH_OK();
  size_t scan_bytes = L.scan_bytes;
  MT_CUDA_OK(cub::DeviceScan::ExclusiveSum(reinterpret_cast<void*>(base + L.scan_tmp), scan_bytes, degp, rowptr_pad,
                                           (int)(N + 1), st));
  count_launch();
  int64_t g = ceil_div<int64_t>(N * 32, 256);
  if (g > (int64_t)kNumSMs * 32) g = (int64_t)kNumSMs * 32;
  if (g < 1) g = 1;
  tc_pad_layout_kernel<<<(unsigned)g, 256, 0, st>>>(rowptr, rowptr_pad, perm, src_sorted, N, orig_pad,
                                                    reinterpret_cast<int32_t*>(base + L.src_pad));
  MT_LAUNCH_OK();
  g = ceil_div<int64_t>(L.cols_max, 256);
  if (g > (int64_t)kNumSMs * 8) g = (int64_t)kNumSMs * 8;
  tc_ypairs_kernel<<<(unsigned)g, 256, 0, st>>>(sh, rowptr_pad, orig_pad, N, y_lmax,
                                                reinterpret_cast<float*>(base + L.ypairs));
  MT_LAUNCH_OK();
  return MT_OK;
}

extern "C" size_t mt_conv_layout_bytes(int y_lmax, int64_t N, int64_t E) {
  if (y_lmax < 0 || y_lmax > MT_LMAX || N <= 0 || E < 0) return 0;
  return tc_layout(y_lmax, N, E).total;
}

extern "C" int mt_conv_layout_prepare(int y_lmax, const void* sh, const int32_t* rowptr, const int32_t* perm,
                                      const int32_t* src_sorted, int64_t N, int64_t E, void* layout,
                                      size_t layout_bytes, mt_stream stream) {
  MT_ENTRY_GUARD();
  MT_REQUIRE(y_lmax >= 0 && y_lmax <= MT_LMAX && N > 0 && E >= 0, "conv layout: bad arguments");
  MT_REQUIRE(E + 3 * N < (int64_t)2147483647, "conv layout: too many edges");
  const TcLayout L = tc_layout(y_lmax, N, E);
  MT_REQUIRE(layout && layout_bytes >= L.total && (reinterpret_cast<uintptr_t>(layout) & 255) == 0,
             "conv layout: buffer of mt_conv_layout_bytes() bytes, 256-byte aligned, required");
  MT_REQUIRE(rowptr && (E == 0 || (sh && perm && src_sorted)), "null pointer");
  return tc_prepare_layout(L, reinterpret_cast<uintptr_t>(layout), y_lmax, static_cast<const float*>(sh), rowptr, perm,
                           src_sorted, N, as_stream(stream));
}

size_t conv_fwd_tc_workspace_bytes(const mt_conv_plan* plan, int64_t N, int64_t E) {
  if (!tc_plan_qualifies(plan) || N <= 0) return 0;
  return tc_workspace_bytes(tc_layout(plan->tc_y_lmax, N, E));
}

static long long* g_tc_dbg = nullptr;  // phase-timing buffer of the next launches (mt_conv_set_debug_buffer)
void conv_fwd_tc_set_debug(void* p) { g_tc_dbg = static_cast<long long*>(p); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    tried = true;
  }
  return fn;
}

// returns MT_OK and sets *used = 1 when the tensor-core path ran; *used = 0 when the plan/shape does not
// qualify (caller falls back to the FMA-pipe kernel)
int conv_fwd_tc_try(const mt_conv_plan* plan, const void* x, const void* sh, const void* emb,
                    const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                    const int32_t* src_sorted, double avg, const void* num_neigh, void* out, void* workspace,
                    size_t workspace_bytes, const void* layout, int64_t N, int64_t E, cudaStream_t st, int* used) {
  *used = 0;
  if (!tc_plan_qualifies(plan)) return MT_OK;
  if (E + 3 * N >= (int64_t)2147483647 || N >= (int64_t)2147483647) return MT_OK;
  const TcLayout L = tc_layout(plan->tc_y_lmax, N, E);
  if (workspace == nullptr || workspace_bytes < tc_workspace_bytes(L)) return MT_OK;
  if ((reinterpret_cast<uintptr_t>(x) & 15) != 0) return MT_OK;
  EncodeTiledFn encode = encode_tiled_fn();
  if (encode == nullptr) return set_error(MT_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.x_dim = plan->x_dim;
  p.y_dim = plan->y_dim;
  p.y_lmax = plan->tc_y_lmax;
  p.out_dim = plan->out_dim;
  p.nl = plan->mlp_num_layers;
  for (int i = 0; i <= p.nl; ++i) p.sizes[i] = plan->mlp_sizes[i];
  for (int i = 0; i < p.nl; ++i) p.w[i] = static_cast<const float*>(mlp_weights[i]);
  p.act = plan->mlp_act;
  p.act_cst = (float)plan->mlp_act_cst;
  p.emb = static_cast<const float*>(emb);
  p.rowptr = rowptr;
  p.perm = perm;
  p.src = src_sorted;
  p.avg = (float)avg;
  p.num_neigh = static_cast<const float*>(num_neigh);
  p.out = static_cast<float*>(out);
  p.N = N;
  p.E = E;
  p.num_parts = plan->tc_num_parts;
  p.dbg = g_tc_dbg;
  {
    const uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255;
    if (layout == nullptr) {  // no per-batch layout from the caller: build it in the workspace
      const int rc = tc_prepare_layout(L, base, plan->tc_y_lmax, static_cast<const float*>(sh), rowptr, perm, src_sorted,
                                       N, st);
      if (rc != MT_OK) return rc;
      layout = reinterpret_cast<const void*>(base);
    }
    const uintptr_t lb = reinterpret_cast<uintptr_t>(layout);
    p.rowptr_pad = reinterpret_cast<int32_t*>(lb + L.rowptr_pad) + (N + 1);
    p.orig_pad = reinterpret_cast<int32_t*>(lb + L.orig_pad);
    p.src_pad = reinterpret_cast<int32_t*>(lb + L.src_pad);
    p.ypairs = reinterpret_cast<float*>(lb + L.ypairs);
    p.hplanes = reinterpret_cast<__nv_bfloat16*>(base + L.total);
    p.cols_max = L.cols_max;
    // hidden layers of the radial MLP, per padded column
    const bool fast = p.nl == 3 && p.sizes[0] <= 8 && p.sizes[1] == kTcK && p.sizes[2] == kTcK && p.act == MT_ACT_SILU;
    int64_t g = ceil_div<int64_t>(L.cols_max, fast ? 256 : 64);
    if (g > (int64_t)kNumSMs * 8) g = (int64_t)kNumSMs * 8;
    if (g < 1) g = 1;
    if (fast) tc_edge_hidden_fast_kernel<<<(unsigned)g, 256, 0, st>>>(p);
    else tc_edge_hidden_kernel<<<(unsigned)g, kHidThreads, 0, st>>>(p);
    MT_LAUNCH_OK();
  }
  // CTAs per part follow the part's cost (every part walks all edges; heavy parts get more SMs)
  int64_t grid = kNumSMs;
  if (grid > N * p.num_parts) grid = N * p.num_parts;
  if (grid < p.num_parts) grid = p.num_parts;
  double cost_sum = 0;
  for (int i = 0; i < p.num_parts; ++i) cost_sum += plan->tc_parts[i].cost > 0 ? plan->tc_parts[i].cost : 1;
  int assigned = 0;
  int lmax = 0;
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  size_t smem_max = 0;
  for (int i = 0; i < p.num_parts; ++i) {
    const mt_conv_tc_part& pt = plan->tc_parts[i];
    TcPartParams& q = p.part[i];
    q.num_tiles = pt.num_tiles;
    q.a_rows = pt.a_rows;
    q.num_bi = pt.num_bi;
    q.x_lo = pt.x_lo;
    q.x_cols = pt.x_cols;
    q.ne = tc_pick_ne(pt, plan->tc_y_lmax);
    for (int k = 0; k < 4; ++k) q.q_count[k] = pt.q_count[k];
    q.row_wcol = pt.row_wcol;
    q.bi_hdr = pt.bi_hdr;
    q.bi_lane = pt.bi_lane;
    q.q_list = pt.q_list;
    const double c = pt.cost > 0 ? pt.cost : 1;
    int n = (i + 1 == p.num_parts) ? (int)grid - assigned : (int)((double)grid * c / cost_sum + 0.5);
    const int left = p.num_parts - 1 - i;
    if (n > (int)grid - assigned - left) n = (int)grid - assigned - left;
    if (n < 1) n = 1;
    if (n > N && N > 0) n = (int)N;
    q.cta_first = assigned;
    q.cta_count = n;
    assigned += n;
    if (pt.lmax > lmax) lmax = pt.lmax;
    const TcSmemLayout L = tc_smem_layout(q.a_rows, q.x_cols, sh_pad_len(p.y_lmax), q.num_bi, q.ne);
    if (L.total > smem_max) smem_max = L.total;
    // x as a 2D tensor [N][x_dim] of fp32, box {x_cols, 1}: tile::gather4 fetches 4 arbitrary rows per instruction
    cuuint64_t dims[2] = {(cuuint64_t)plan->x_dim, (cuuint64_t)(N > 0 ? N : 1)};
    cuuint64_t strides[1] = {(cuuint64_t)plan->x_dim * 4};
    cuuint32_t box[2] = {(cuuint32_t)q.x_cols, 1};
    cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&maps.m[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(x), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(MT_ECUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    // the h planes [3 planes x 4 k-groups][cols_max][16 bytes] as a 3D byte tensor, box {16, NE, 12}: a chunk's twelve
    // plane segments in one TMA instruction, landing as the dense [12][NE][16 B] B operand
    cuuint64_t hdims[3] = {16, (cuuint64_t)p.cols_max, 12};
    cuuint64_t hstrides[2] = {16, (cuuint64_t)p.cols_max * 16};
    cuuint32_t hbox[3] = {16, (cuuint32_t)q.ne, 12};
    cuuint32_t hestr[3] = {1, 1, 1};
    const CUresult rh = encode(&maps.h[i], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, p.hplanes, hdims, hstrides, hbox, hestr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rh != CUDA_SUCCESS) return set_error(MT_ECUDA, "cuTensorMapEncodeTiled (h planes) failed (%d)", (int)rh);
  }
  grid = assigned;
  static thread_local size_t configured[2] = {0, 0};
  const int vi = lmax <= 2 ? 0 : 1;
  if (smem_max > configured[vi]) {
    if (vi == 0)
      MT_CUDA_OK(cudaFuncSetAttribute(conv_fwd_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemLimit));
    else
      MT_CUDA_OK(cudaFuncSetAttribute(conv_fwd_tc_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemLimit));
    configured[vi] = kTcSmemLimit;
  }
  if (vi == 0) conv_fwd_tc_kernel<2><<<(unsigned)grid, kTcThreads, smem_max, st>>>(p, maps);
  else conv_fwd_tc_kernel<4><<<(unsigned)grid, kTcThreads, smem_max, st>>>(p, maps);
  MT_LAUNCH_OK();
  *used = 1;
  return MT_OK;
}

}  // namespace mt
