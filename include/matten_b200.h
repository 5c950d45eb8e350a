/*
 * matten_b200 -- C ABI of the B200-native (sm_100a) equivariant message-passing
 * hot path of MatTen (wengroup/matten).
 *
 * Drop-in boundary.  The reference is pure Python; the arithmetic on this path
 * lives in e3nn 0.5.1 / torch_scatter, called from src/matten/nn/*.py.  Every
 * entry point below replaces one of those call sites (cited per function) and is
 * what a `ctypes` / `torch.library` binding on the reference side binds (see
 * INTEGRATION.md).  Conventions:
 *
 *   - plain device pointers + sizes; the caller owns every buffer (inputs,
 *     outputs, workspaces) and allocates them with whatever allocator it uses
 *     (torch in our host layer).  The library never allocates on the hot path
 *     and never synchronises the stream;
 *   - all work is enqueued on the `stream` argument (a cudaStream_t passed as
 *     void*); any number of host threads may call concurrently;
 *   - `dtype` selects the arithmetic type of every `void*` tensor of the call:
 *     MT_F32 or MT_F64 (the reference's DTYPE, src/matten/data/_dtype.py:3);
 *   - tensors are dense row-major; index tensors coming from the reference's
 *     graph dict are int64 (src/matten/data/_dtype.py:4); bookkeeping produced
 *     by this library (CSR row pointers, permutations) is int32;
 *   - return value: MT_OK (0) or a negative mt_status; mt_last_error() returns a
 *     thread-local message.  Nothing throws or exits across the boundary;
 *   - data errors that can only be seen on the device (atomic number not in the
 *     model's species list, unsorted batch vector, index out of range) are
 *     OR-ed into a caller-provided int32 device flag word (`err_flag`, may be
 *     NULL) so that no call has to synchronise; the caller reads it once per
 *     batch (bits: MT_FLAG_*).
 *   - there is NO CPU fallback: on a device that is not compute capability 10.x
 *     every compute entry point returns MT_EARCH.
 */
#ifndef MATTEN_B200_H
#define MATTEN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MT_ABI_VERSION 2
#define MT_MAX_MLP_LAYERS 6
#define MT_LMAX 4

typedef enum {
  MT_OK = 0,
  MT_EINVAL = -1, /* bad argument / unsupported configuration */
  MT_EARCH = -2,  /* device is not sm_100 */
  MT_ECUDA = -3   /* CUDA runtime error (message in mt_last_error) */
} mt_status;

typedef enum { MT_F32 = 0, MT_F64 = 1 } mt_dtype;

/* activation ids (reference src/matten/nn/utils.py:14-26) */
typedef enum {
  MT_ACT_NONE = 0,
  MT_ACT_SILU = 1,
  MT_ACT_TANH = 2,
  MT_ACT_SIGMOID = 3,
  MT_ACT_SSP = 4, /* shifted softplus, src/matten/nn/_nequip.py:17-39 */
  MT_ACT_ABS = 5
} mt_act;

/* bits of the device error flag word */
#define MT_FLAG_BAD_SPECIES 1 /* atomic number outside the allowed list   */
#define MT_FLAG_BAD_INDEX 2   /* edge / key index out of range            */
#define MT_FLAG_UNSORTED 4    /* batch vector not non-decreasing          */

typedef void* mt_stream; /* cudaStream_t */

int mt_abi_version(void);
const char* mt_last_error(void);
/* Number of kernels this library has launched in this process (all threads). */
uint64_t mt_launch_count(void);
/* MT_OK if `device` is compute capability 10.x, else MT_EARCH. */
int mt_device_supported(int device);

/* ------------------------------------------------------------------------- *
 * Edge geometry.
 * ------------------------------------------------------------------------- */

/* a1: with_edge_vectors, reference src/matten/nn/_nequip.py:214-268.
 *   vec[e] = pos[ei[1,e]] - pos[ei[0,e]] + shift[e] @ cell[batch[ei[0,e]]]
 *   len[e] = |vec[e]|
 * pos [N,3]; edge_index [2,E] int64; shift [E,3] and cell [B,3,3] may both be NULL
 * (no periodic images); batch [N] int64 may be NULL when B == 1.
 * edge_vec [E,3] and edge_len [E] are outputs (either may be NULL). */
int mt_edge_vectors(int dtype, const void* pos, const int64_t* edge_index,
                    const void* edge_cell_shift, const void* cell, const int64_t* batch,
                    int64_t N, int64_t E, int64_t B, void* edge_vec, void* edge_len,
                    int32_t* err_flag, mt_stream stream);

/* a2: e3nn.o3.SphericalHarmonics(0..lmax, normalize=True, 'component'), reference
 * src/matten/nn/_nequip.py:167-176.  edge_vec [E,3] -> edge_sh [E,(lmax+1)^2].
 * normalize != 0 divides by the length first (the reference always does). */
int mt_edge_sh(int dtype, const void* edge_vec, int64_t E, int lmax, int normalize,
               void* edge_sh, mt_stream stream);

/* a3 / a3': radial basis of the edge length, edge_len [E] -> edge_emb [E,num_basis].
 *  mode 0: e3nn.math.soft_one_hot_linspace(x, start, end, n, 'bessel', cutoff) * sqrt(n)
 *          (EdgeLengthEmbedding, reference src/matten/nn/embedding.py:185-203);
 *  mode 1: BesselBasis(r_max=end) * PolynomialCutoff(r_max=end, p)  (RadialBasisEdge-
 *          Encoding, reference src/matten/nn/_nequip.py:43-126,180-210); bessel_w [n]
 *          holds the (trainable) frequencies, NULL means n*pi;
 *  mode 2: d(mode 1)/d bessel_w[k] per (edge, k) -- the frequency gradient is its column-wise
 *          product sum with the incoming gradient (mt_col_reduce);
 *  modes 3-6: e3nn.math.soft_one_hot_linspace(x, start, end, n, basis, cutoff) * sqrt(n) with basis
 *          3 'gaussian', 4 'cosine', 5 'smooth_finite', 6 'fourier' (EdgeLengthEmbedding with that
 *          basis).  Modes 3-5 without cutoff need n >= 2 (their centres are linspace(start, end, n)).
 *  poly_p and bessel_w are read by modes 1 and 2 only; cutoff by modes 0 and 3-6. */
int mt_edge_radial(int dtype, const void* edge_len, int64_t E, int mode, int num_basis,
                   double start, double end, int cutoff, double poly_p, const void* bessel_w,
                   void* edge_emb, mt_stream stream);

/* Backward of the edge geometry (first derivatives only), what autograd does in the reference through
 * with_edge_vectors, SphericalHarmonics and the radial bases.  Deterministic: no float atomics.
 *
 * Backward of a2 (reference src/matten/nn/_nequip.py:167-176): grad_vec[e] = J_Y(vec[e])^T grad_sh[e], including
 * the v / max(|v|, 1e-12) normalisation when normalize != 0.  grad_sh [E,(lmax+1)^2] -> grad_vec [E,3]. */
int mt_edge_sh_bwd(int dtype, const void* edge_vec, const void* grad_sh, int64_t E, int lmax, int normalize,
                   void* grad_vec, mt_stream stream);

/* Backward of a3 / a3' with respect to the length (reference src/matten/nn/embedding.py:185-203 for modes 0 and
 * 3-6, src/matten/nn/_nequip.py:43-126 for mode 1): grad_len[e] = sum_k grad_emb[e,k] d edge_emb[e,k] / d len[e],
 * the k-sum in order.  Arguments as in mt_edge_radial (mode 0, 1 or 3-6); grad_emb [E,num_basis] -> grad_len [E].
 * The masks of modes 0, 4 and 6 and the r < end factor of mode 1 have zero derivative; for mode 5 the derivative
 * of exp(-1/t) is taken as 0 wherever exp(-1/t) is 0. */
int mt_edge_radial_bwd(int dtype, const void* edge_len, const void* grad_emb, int64_t E, int mode, int num_basis,
                       double start, double end, int cutoff, double poly_p, const void* bessel_w, void* grad_len,
                       mt_stream stream);

/* Backward of a1 (reference src/matten/nn/_nequip.py:214-268):
 *   dv[e]          = grad_vec[e] + grad_len[e] vec[e] / |vec[e]|     (0 for the length term where |vec[e]| = 0)
 *   grad_pos[n]    = sum_{ei[1,e] = n} dv[e] - sum_{ei[0,e] = n} dv[e]
 *   grad_cell[g]  += shift[e] (x) dv[e]  over the edges whose sender is in graph g
 * edge_vec [E,3] is the forward's output; grad_vec [E,3] and grad_len [E] may be NULL (no gradient).  The sums run
 * over the receiver CSR (rowptr [N+1], perm [E] of mt_csr_by_key on edge_index[1]) and the sender CSR of the
 * receiver-sorted list (sender_ptr [N+1], sender_perm [E], as for mt_conv_bwd), in CSR order.  graph_ptr [B+1] int32
 * (first node of every graph; nodes of a graph contiguous) may be NULL when B == 1.  edge_cell_shift [E,3] may be NULL
 * (no periodic images); then grad_cell must be NULL.  Outputs grad_pos [N,3] and grad_cell [B,3,3] (either may be
 * NULL).  workspace: mt_edge_vectors_bwd_workspace_bytes bytes. */
size_t mt_edge_vectors_bwd_workspace_bytes(int dtype, int64_t E, int64_t B);
int mt_edge_vectors_bwd(int dtype, const void* edge_vec, const void* grad_vec, const void* grad_len,
                        const void* edge_cell_shift, const int32_t* rowptr, const int32_t* perm,
                        const int32_t* sender_ptr, const int32_t* sender_perm, const int32_t* graph_ptr, int64_t N,
                        int64_t E, int64_t B, void* grad_pos, void* grad_cell, void* workspace,
                        size_t workspace_bytes, mt_stream stream);

/* ------------------------------------------------------------------------- *
 * Index bookkeeping (bit-exact integer work).
 * ------------------------------------------------------------------------- */

/* Stable counting sort of E int64 keys in [0, num_keys): the receiver-sorted CSR
 * that replaces torch_scatter's atomics (reference src/matten/nn/conv.py:114), and
 * the species grouping used by the species-indexed linears.
 *   rowptr [num_keys+1]: rowptr[k] = #keys < k;  perm [E]: perm[i] = original index of
 *   the i-th entry in sorted order (ties in ascending original index).
 * perm may be NULL (row pointers only, e.g. graph pointers from the batch vector).
 * workspace: mt_csr_workspace_bytes(num_keys, E) bytes. */
size_t mt_csr_workspace_bytes(int64_t num_keys, int64_t E);
int mt_csr_by_key(const int64_t* keys, int64_t E, int64_t num_keys, int32_t* rowptr,
                  int32_t* perm, void* workspace, size_t workspace_bytes, int32_t* err_flag,
                  mt_stream stream);

/* out[i] = (int32) src[perm[i]]  (perm NULL: identity). */
int mt_gather_i64_to_i32(const int64_t* src, const int32_t* perm, int64_t n, int32_t* out,
                         mt_stream stream);

/* Sets MT_FLAG_UNSORTED if keys is not non-decreasing. */
int mt_check_sorted(const int64_t* keys, int64_t n, int32_t* err_flag, mt_stream stream);

/* a16 (SURVEY section 8f rank 1): periodic neighbour list of a batch of crystals on the GPU.  Replaces
 * neighbor_list_and_relative_vec (reference src/matten/data/data.py:285-413: ASE primitive_neighbor_list("ijS",
 * self_interaction=True) minus the true self edges).  Every ordered pair (i, j, S) of one crystal with
 * |pos[j] - pos[i] + S @ cell| < r_max except (i == j, S == 0); all arithmetic in fp64 whatever `dtype` is; edges in
 * the canonical order (i, j, Sx, Sy, Sz).  Two calls, because the edge count is data dependent:
 *   mt_neighbor_count: offsets [N+1] = exclusive scan of the per-centre neighbour counts, offsets[N] = E
 *                      (the caller reads offsets[N] to size the outputs: the one synchronisation of graph building);
 *   mt_neighbor_fill : edge_index [2,E] int64 (row 0 = centre i, row 1 = neighbour j), edge_cell_shift [E,3] and
 *                      num_neigh [N] (may be NULL) in `dtype` (the reference stores both as floats).
 * pos [N,3], cell [B,3,3] in `dtype`; batch [N] int64 (NULL when B == 1); ptr [B+1] int64 node offsets of the graphs.
 * workspace: mt_neighbor_workspace_bytes(N, B), shared by the two calls. */
size_t mt_neighbor_workspace_bytes(int64_t N, int64_t B);
int mt_neighbor_count(int dtype, const void* pos, const void* cell, const int64_t* batch, const int64_t* ptr,
                      int64_t N, int64_t B, double r_max, int32_t* offsets, void* workspace, size_t workspace_bytes,
                      mt_stream stream);
int mt_neighbor_fill(int dtype, const void* pos, const int64_t* batch, const int64_t* ptr, int64_t N, int64_t B,
                     double r_max, const int32_t* offsets, const void* workspace, int64_t* edge_index,
                     void* edge_cell_shift, void* num_neigh, int64_t E, mt_stream stream);

/* a4: _AtomicNumberToIndex + one-hot + Linear(S, dim, bias), reference
 * src/matten/nn/embedding.py:85-110, 206-263.
 *   idx = lut[Z - min_Z] (MT_FLAG_BAD_SPECIES if Z out of range or lut == -1)
 *   node_attrs[n, :] = one_hot(idx, S);  node_feats[n, j] = lin_w[j, idx] + lin_b[j]
 * atomic_numbers may be NULL when species_index (in/out, int64 [N]) is already given
 * (z_given == 0). Any output may be NULL. lin_w is [dim, S] (torch Linear layout). */
int mt_species_embed(int dtype, const int64_t* atomic_numbers, int z_given, const int64_t* lut,
                     int64_t min_z, int64_t max_z, int num_species, int dim, const void* lin_w,
                     const void* lin_b, int64_t N, int64_t* species_index, void* node_attrs,
                     void* node_feats, int32_t* err_flag, mt_stream stream);

/* ------------------------------------------------------------------------- *
 * a6 + a7: fused  radial MLP -> uvu tensor product -> segmented sum over the
 * receiver's edges -> / sqrt(#neighbours).  Replaces weight_nn + tp + scatter + div
 * of reference src/matten/nn/conv.py:113-120 and src/matten/nn/utils.py:255-263.
 * Per-edge weights and messages never touch HBM.
 * ------------------------------------------------------------------------- */

/* The "plan" is a set of small int32 device tables built by the host once per
 * layer (matten_b200/plan.py: the uvu instruction list of reference
 * src/matten/nn/utils.py:205-237 regrouped into warp work items by (l1,l2,l3)).
 *   item_hdr  [num_items,2]  : {cg_type_id, cols_per_warp (power of two <= 32)}
 *   slot_tab  [num_items,32,4]: per lane {weight column (-1 = idle lane), offset of
 *                              x[u,:] in the x row, offset of the sh block, offset of
 *                              out[u,:] in the output row}
 * mlp: num_layers weight matrices, weights[i] is [sizes[i], sizes[i+1]] row-major (the
 * e3nn FullyConnectedNet layout), applied as act(x @ W / sqrt(sizes[i])) * act_cst on
 * all but the last layer; sizes[num_layers] == weight_numel of the tensor product. */
#define MT_TC_MAX_PARTS 4
#define MT_TC_MAX_BI 64
/* One part of the tcgen05 plan (device tables, int32):
 *   row_wcol [num_tiles*128] : weight column held by every A row / TMEM lane (-1 = zero row)
 *   bi_hdr   [num_bi,8]      : {bundle id (csrc/generated/cg_bundles.cuh), mode (0 = lane per channel, 1 = 16x256b
 *                              edge phases), channels per row block, active-path mask, quarter, slot of path 0 / 1 / 2
 *                              (2 * tile + half)}
 *   bi_lane  [num_bi,32,4]   : per lane {offset of x[u,:] inside the part's window, out offset of path 0 / 1 / 2
 *                              (-1 = this lane stores nothing for the path)}
 *   q_list   [4,MT_TC_MAX_BI], q_count[4]: bundle instances of every quarter (32 TMEM lanes = one warp
 *                              scheduler), heaviest first */
typedef struct {
  int32_t num_tiles;
  int32_t a_rows;       /* A rows kept in shared memory: a multiple of 32 above the last used row */
  int32_t num_bi;
  int32_t x_lo, x_cols; /* window of the x row this part gathers (floats; multiples of 4 / 8) */
  int32_t lmax;         /* largest degree among its bundles (selects the kernel instantiation) */
  int32_t cost;         /* relative cost: share of the CTAs */
  int32_t q_count[4];
  const int32_t* row_wcol; /* device */
  const int32_t* bi_hdr;   /* device */
  const int32_t* bi_lane;  /* device */
  const int32_t* q_list;   /* device */
} mt_conv_tc_part;

typedef struct {
  int32_t x_dim;        /* row length of x (node features)          */
  int32_t y_dim;        /* row length of sh (edge attrs)            */
  int32_t out_dim;      /* row length of the output (irreps_mid)    */
  int32_t num_items;    /* warp work items                          */
  const int32_t* item_hdr; /* device */
  const int32_t* slot_tab; /* device */
  int32_t mlp_num_layers;
  int32_t mlp_sizes[MT_MAX_MLP_LAYERS + 1];
  int32_t mlp_act;      /* mt_act of the hidden layers              */
  double mlp_act_cst;   /* normalize2mom constant of that activation */
  /* Optional tables of the tcgen05 path (fp32, MLP layer sizes <= 32, <= 2 hidden layers); tc_num_parts == 0
   * disables it.  Built by matten_b200/tcplan.py (vocabulary there): the weight columns are rows of the MMA A
   * operand = lanes of tensor memory; a *bundle instance* is a group of input channels x a compile-time list
   * of (l2, l3) paths sharing the loads of x[u, :] and of the edge's spherical harmonics; a *part* owns <= 4
   * tiles of 128 rows and a window of the x row (layers whose weights exceed 512 rows are cut into parts). */
  int32_t tc_num_parts;
  int32_t tc_y_lmax;    /* edge attrs are the harmonics 0 .. tc_y_lmax, one block each, in order */
  mt_conv_tc_part tc_parts[MT_TC_MAX_PARTS];
  /* Tables of the backward pass (mt_conv_bwd), organised by INPUT channel so that the gradient of a
   * gathered x row is a register sum in fixed path order; bw_num_items == 0: forward-only plan.
   *   bw_item_hdr [bw_num_items,4]   : {l1, cols_per_warp, first path, path count}
   *   bw_lane_tab [bw_num_items,32,2]: per lane {u (-1 = idle lane), offset of x[u,:] in the x row}
   *   bw_path_tab [bw_num_paths,4]   : {cg_type_id, weight column of u = 0, sh offset, out offset of u = 0} */
  int32_t bw_num_items;
  int32_t bw_num_paths;
  const int32_t* bw_item_hdr; /* device */
  const int32_t* bw_lane_tab; /* device */
  const int32_t* bw_path_tab; /* device */
} mt_conv_plan;

/* x [N,x_dim]; sh [E,y_dim], emb [E,mlp_sizes[0]] in ORIGINAL edge order;
 * rowptr [N+1], perm [E], src_sorted [E] from mt_csr_by_key / mt_gather_i64_to_i32 on
 * edge_index[1] / edge_index[0].  out [N,out_dim] =
 *   (sum_{e: dst(e)=n} msg_e) / sqrt(avg_num_neighbors)        if num_neigh == NULL
 *   (sum ...)             / sqrt(num_neigh[n])                  otherwise (reference
 *   src/matten/nn/conv.py:116-120). Summation order is the CSR order: deterministic. */
/* workspace (bytes) of the tcgen05 path: room for the per-batch edge layout of mt_conv_layout_prepare, which a call
 * without `layout` builds there, and the last hidden activation of the radial MLP as bf16 hi/mid/lo planes (192 B per
 * column).  0 when the plan / dtype runs on the FMA-pipe kernel, which needs none. */
size_t mt_conv_fwd_workspace_bytes(const mt_conv_plan* plan, int dtype, int64_t N, int64_t E);
int mt_conv_fwd(const mt_conv_plan* plan, int dtype, const void* x, const void* sh,
                const void* emb, const void* const* mlp_weights, const int32_t* rowptr,
                const int32_t* perm, const int32_t* src_sorted, double avg_num_neighbors,
                const void* num_neigh, void* out, void* workspace, size_t workspace_bytes,
                const void* layout, int64_t N, int64_t E, mt_stream stream);

/* The layer-invariant inputs of the tcgen05 path: the padded column order of the receiver-sorted edge list and the
 * pair-interleaved spherical-harmonics rows.  Every PointConv layer of a forward shares the graph and edge_sh
 * (reference src/matten/model_factory/tfn_scalar_tensor.py:160-214: one spharm_edges module feeds all layers), so the
 * caller prepares them ONCE per batch and passes the buffer as `layout` to every mt_conv_fwd of that batch
 * (layout NULL: mt_conv_fwd builds the same layout in its workspace at every call).  fp32 only (the fp64 and FMA-pipe
 * kernels ignore it); y_lmax is the largest degree of edge_sh, whose blocks must be 0 .. y_lmax in order.
 * layout: mt_conv_layout_bytes(y_lmax, N, E) bytes, 256-byte aligned. */
size_t mt_conv_layout_bytes(int y_lmax, int64_t N, int64_t E);
int mt_conv_layout_prepare(int y_lmax, const void* sh, const int32_t* rowptr, const int32_t* perm,
                           const int32_t* src_sorted, int64_t N, int64_t E, void* layout, size_t layout_bytes,
                           mt_stream stream);

/* Which fp32 kernel mt_conv_fwd uses: 0 = automatic (tcgen05 when the plan qualifies, else FMA pipes), 1 = tcgen05
 * only (MT_EINVAL when the plan does not qualify), 2 = FMA pipes only.  Process-wide, initially 0.  Returns the
 * previous setting. */
int mt_conv_select_impl(int impl);
/* Profiling aid: device buffer of >= 32 * 8 int64 that receives the per-warp phase timings (clock64 sums, slot
 * meanings in csrc/conv_fwd_tc.cuh) of CTA 0 of every following tcgen05 launch; NULL (default) turns it off. */
void mt_conv_set_debug_buffer(void* device_buffer);

/* Backward of mt_conv_fwd (what autograd does through weight_nn + tp + scatter + div in the reference,
 * src/matten/nn/conv.py:111-120).  Inputs as in mt_conv_fwd plus
 *   grad_out [N,out_dim]            : dL/d out
 *   sender_ptr [N+1], sender_perm [E]: CSR over the SENDERS of the receiver-sorted edge list
 *                                     (mt_csr_by_key on src_sorted): sender_perm[i] is a position in the
 *                                     receiver-sorted list
 * Outputs (either group may be NULL to skip it):
 *   grad_x [N,x_dim]                : dL/dx, summed per sender in sender-CSR order (deterministic)
 *   grad_mlp_weights[i]             : dL/d weights[i], same shapes as mlp_weights[i]; per-CTA partial sums
 *                                     reduced in a fixed order (deterministic for a fixed N, E)
 * workspace: mt_conv_bwd_workspace_bytes bytes (hidden pre-activations, per-edge dw / dx scratch, partial
 * weight gradients). */
size_t mt_conv_bwd_workspace_bytes(const mt_conv_plan* plan, int dtype, int64_t N, int64_t E);
int mt_conv_bwd(const mt_conv_plan* plan, int dtype, const void* x, const void* sh, const void* emb,
                const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                const int32_t* src_sorted, const int32_t* sender_ptr, const int32_t* sender_perm,
                double avg_num_neighbors, const void* num_neigh, const void* grad_out, void* grad_x,
                void* const* grad_mlp_weights, void* workspace, size_t workspace_bytes, int64_t N, int64_t E,
                mt_stream stream);
/* mt_conv_bwd plus the gradients with respect to the edge inputs (reference src/matten/nn/utils.py:260-263, the
 * sh and edge_embedding arguments of tp(x[src], sh, weight_nn(edge_embedding))), in the caller's edge order:
 *   grad_sh  [E,y_dim]        : dL/d sh
 *   grad_emb [E,mlp_sizes[0]] : dL/d edge_embedding
 * Either may be NULL; with both NULL this is mt_conv_bwd.  Same workspace as mt_conv_bwd. */
int mt_conv_bwd_full(const mt_conv_plan* plan, int dtype, const void* x, const void* sh, const void* emb,
                     const void* const* mlp_weights, const int32_t* rowptr, const int32_t* perm,
                     const int32_t* src_sorted, const int32_t* sender_ptr, const int32_t* sender_perm,
                     double avg_num_neighbors, const void* num_neigh, const void* grad_out, void* grad_x,
                     void* const* grad_mlp_weights, void* grad_sh, void* grad_emb, void* workspace,
                     size_t workspace_bytes, int64_t N, int64_t E, mt_stream stream);

/* ------------------------------------------------------------------------- *
 * a8 / a11 / a13 / a14: irreps-wise linear maps.
 *   FullyConnectedTensorProduct(x, one_hot(species), out)  (reference
 *   src/matten/nn/conv.py:59-61,77-79,84-86)  ==  species-indexed linear;
 *   e3nn.o3.Linear (reference src/matten/nn/nodewise.py:111,
 *   model_factory/tfn_scalar_tensor.py:50) is the num_species == 1 case, and
 *   CartesianTensor.to_cartesian (reference src/matten/utils.py:123-124) is a single
 *   dense block.
 * For each block b:  out[n, out_off + w*dim + m] (+)= scale *
 *        sum_u weight[w_off + (u*S + s_n)*mul_out + w] * x[n, in_off + u*dim + m]
 * A block with mul_in == 0 zero-fills its output range (irreps with no path).
 * dim must be 2l+1 for l <= 4 (1, 3, 5, 7 or 9); mt_linear_fwd and mt_linear_bwd return
 * MT_EINVAL for any other dim, and for a block outside in_dim / out_dim, before any launch.
 * ------------------------------------------------------------------------- */
typedef struct {
  int32_t in_off, out_off, mul_in, mul_out, dim, w_off;
  double scale;
} mt_lin_block;

/* species_perm [N] / species_ptr [S+1]: nodes grouped by species (mt_csr_by_key on
 * species_index); both NULL when num_species == 1.  accumulate != 0 adds into out. */
int mt_linear_fwd(int dtype, const mt_lin_block* blocks, int num_blocks, int in_dim,
                  int out_dim, int num_species, const void* x, const void* weight,
                  const int32_t* species_perm, const int32_t* species_ptr, int accumulate,
                  void* out, int64_t N, mt_stream stream);

/* Backward of mt_linear_fwd.
 *   grad_x [N,in_dim]  (may be NULL): scale * sum_w weight[(u*S+s_n)*mul_out + w] * grad_out[n, w, m];
 *                      elements of x that feed no block get 0.  accumulate_x != 0 adds into grad_x.
 *   grad_w [weight numel] (may be NULL): scale * sum_{n of species s} sum_m x[n,u,m] * grad_out[n,w,m];
 *                      node range split over CTAs, partials reduced in fixed order (deterministic).
 *                      accumulate_w != 0 adds into grad_w (gradient accumulation).
 * workspace: mt_linear_bwd_workspace_bytes(weight_numel) bytes (0 when grad_w is NULL). */
size_t mt_linear_bwd_workspace_bytes(int dtype, int64_t weight_numel);
int mt_linear_bwd(int dtype, const mt_lin_block* blocks, int num_blocks, int in_dim, int out_dim,
                  int num_species, int64_t weight_numel, const void* x, const void* weight,
                  const void* grad_out, const int32_t* species_perm, const int32_t* species_ptr,
                  void* grad_x, int accumulate_x, void* grad_w, int accumulate_w, void* workspace,
                  size_t workspace_bytes, int64_t N, mt_stream stream);

/* ------------------------------------------------------------------------- *
 * a9 + a10: e3nn.nn.Gate followed by e3nn.nn.BatchNorm in eval mode (reference
 * src/matten/nn/utils.py:134-140, 418, applied at src/matten/nn/conv.py:209-211).
 * Per OUTPUT element j (tables are device arrays of length out_dim):
 *   v = x[n, src_idx[j]]
 *   gate_idx[j] <  0 : y = act_id[j](v) * act_cst[j]                 (scalar)
 *   gate_idx[j] >= 0 : y = v * act_id[j](x[n, gate_idx[j]]) * act_cst[j]  (gated)
 *   out[n,j] = y * affine_a[j] + affine_b[j]      (affine_* NULL: identity)
 * ------------------------------------------------------------------------- */
int mt_gate_fwd(int dtype, const void* x, int in_dim, int out_dim, const int32_t* src_idx,
                const int32_t* gate_idx, const int32_t* act_id, const void* act_cst,
                const void* affine_a, const void* affine_b, void* out, int64_t N,
                mt_stream stream);

/* Backward of mt_gate_fwd w.r.t. x (the affine is treated as constant).  inv_first / inv_count
 * [in_dim] invert the element tables: input i feeds outputs inv_first[i] .. + inv_count[i] - 1 (one
 * output for a scalar or gated element, the 2l+1 gated outputs for a gate; count 0: unused input). */
int mt_gate_bwd(int dtype, const void* x, const void* grad_out, int in_dim, int out_dim,
                const int32_t* src_idx, const int32_t* gate_idx, const int32_t* act_id, const void* act_cst,
                const void* affine_a, const int32_t* inv_first, const int32_t* inv_count, void* grad_x,
                int64_t N, mt_stream stream);

/* Column reductions over the node axis (training-mode e3nn BatchNorm statistics and their backward,
 * reference src/matten/nn/utils.py:418; bias gradients):
 *   out[j] = sum_n (a[n,j] - shift_a[j]) * (b ? (b[n,j] - shift_b[j]) : 1)      j < dim
 * a, b [N,dim] (b may be NULL or equal to a); shift_* [dim] may be NULL (0).  Two-stage, fixed order.
 * workspace: mt_col_reduce_workspace_bytes(dtype, dim) bytes. */
size_t mt_col_reduce_workspace_bytes(int dtype, int dim);
int mt_col_reduce(int dtype, const void* a, const void* shift_a, const void* b, const void* shift_b,
                  int64_t N, int dim, void* out, void* workspace, size_t workspace_bytes, mt_stream stream);

/* out[n,j] = ca[j] * a[n,j] + (b ? cb[j] * b[n,j] : 0) + cc[j]   (BatchNorm apply and its backward). */
int mt_affine2(int dtype, const void* a, const void* ca, const void* b, const void* cb, const void* cc,
               void* out, int64_t N, int dim, mt_stream stream);

/* Backward of mt_segment_reduce for mode 0 (sum) / 1 (mean): grad_x[n,:] = grad_out[b(n),:] (/ count). */
int mt_segment_reduce_bwd(int dtype, const void* grad_out, const int32_t* ptr, int dim, int64_t B, int64_t N,
                          int mode, void* grad_x, mt_stream stream);

/* out[s,:] = sum_{i in [ptr[s], ptr[s+1])} x[perm ? perm[i] : i, :], fixed order; num_rows = ptr[num_segments]
 * (a block-level sum is used when segments are long).  Used for the species-embedding gradient (backward of mt_species_embed: dW[:,s]) and for the
 * per-sender reduction of the conv backward. */
int mt_segment_sum_gather(int dtype, const void* x, const int32_t* perm, const int32_t* ptr, int dim,
                          int64_t num_segments, int64_t num_rows, void* out, mt_stream stream);

/* a17: loss and optimiser (reference src/matten/model/model.py:234-274: MSE with mean reduction;
 * scripts/configs/materials_tensor.yaml:103-107: torch.optim.Adam(lr, weight_decay), L2 form).
 *   mt_mse_loss: loss[0] = mean((pred - target)^2), grad[i] = 2 (pred - target) / n * grad_scale
 *                (either output may be NULL); single CTA, fixed order.
 *   mt_adam_step: p, g, m, v flat [n]; torch.optim.Adam semantics (amsgrad off):
 *                g' = g * grad_scale + wd * p; m = b1 m + (1-b1) g'; v = b2 v + (1-b2) g'^2;
 *                p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps) */
int mt_mse_loss(int dtype, const void* pred, const void* target, int64_t n, double grad_scale, void* loss,
                void* grad, mt_stream stream);
int mt_adam_step(int dtype, void* p, const void* g, void* m, void* v, int64_t n, double lr, double beta1,
                 double beta2, double eps, double weight_decay, double grad_scale, int64_t step,
                 mt_stream stream);

/* a12: torch_scatter.scatter(x, batch, reduce) over a SORTED batch vector (reference
 * src/matten/nn/nodewise.py:142-148).  ptr [B+1] from mt_csr_by_key on batch.
 * mode: 0 sum, 1 mean, 2 min, 3 max.  x [N,dim] -> out [B,dim]. */
int mt_segment_reduce(int dtype, const void* x, const int32_t* ptr, int dim, int64_t B,
                      int mode, void* out, mt_stream stream);

/* Backward of mt_segment_reduce for mode 2 (min) / 3 (max): the gradient of a segment's column goes to the first
 * row holding the extreme value, every other row of the segment gets 0 (torch_scatter's arg-based backward).
 * x [N,dim] is the forward input; grad_x [N,dim] must cover exactly the rows ptr spans. */
int mt_segment_extreme_bwd(int dtype, const void* x, const void* grad_out, const int32_t* ptr, int dim, int64_t B,
                           int mode, void* grad_x, mt_stream stream);

/* f4: graph-wise InstanceNorm (reference src/matten/nn/utils.py:448-588, ``NormalizationLayer(method="instance")``
 * at :421-426).  Every graph is an instance, its nodes the samples.  Channel c (one copy of one irrep) owns the
 * columns [chan_first[c], chan_first[c] + chan_dim[c]); chan_scalar[c] is the index among the l = 0 channels (either
 * parity, as the reference tests ``ir.l == 0``) or -1.  l = 0 channels are centred by the graph mean; the squared
 * norm is averaged (normalization 0, "component") or summed (1, "norm") over the 2l+1 components, then reduced over
 * the graph's nodes by mean (reduce 0) or max (1); y = (x - mean) * (v + eps)^-1/2 * weight[c] (+ bias[scalar]).
 * The same statistics are used in training and evaluation, as in the reference.  graph_ptr [G+1] spans the nodes of
 * each graph (sorted batch vector).  weight [num_channels] / bias [num_scalar] may be NULL (affine=False).
 * save_mean, save_rstd [G,num_channels] (always double: the statistics are evaluated in double for either dtype,
 * centring subtracts nearly equal numbers) and save_arg [G,num_channels] (row chosen by the max reduce) feed
 * the backward.  Backward: grad_x [N,dim]; grad_weight_part / grad_bias_part [G,num_channels] per-graph partial
 * sums (either may be NULL) that the caller adds over graphs with mt_col_reduce. */
int mt_instance_norm_fwd(int dtype, const void* x, const int32_t* graph_ptr, int64_t G, int dim, int num_channels,
                         const int32_t* chan_first, const int32_t* chan_dim, const int32_t* chan_scalar,
                         const void* weight, const void* bias, double eps, int reduce, int normalization, void* out,
                         void* save_mean, void* save_rstd, int32_t* save_arg, mt_stream stream);
int mt_instance_norm_bwd(int dtype, const void* x, const void* grad_out, const int32_t* graph_ptr, int64_t G, int dim,
                         int num_channels, const int32_t* chan_first, const int32_t* chan_dim,
                         const int32_t* chan_scalar, const void* weight, int reduce, int normalization,
                         const void* save_mean, const void* save_rstd, const int32_t* save_arg, void* grad_x,
                         void* grad_weight_part, void* grad_bias_part, mt_stream stream);

/* f4: e3nn.nn.NormActivation(irreps, f, normalize=True, epsilon=1e-8, bias=False) as the reference builds it
 * (src/matten/nn/utils.py:142-150, ``activation_type="norm"``): per channel n = sqrt(max(sum_m x_m^2, epsilon^2)),
 * y_m = x_m * f(n) / n with f the raw activation act_id (MT_ACT_*, no second-moment constant).  The backward
 * treats a clamped norm as a constant, as autograd does for the masked assignment. */
int mt_norm_act_fwd(int dtype, const void* x, int dim, int num_channels, const int32_t* chan_first,
                    const int32_t* chan_dim, int act_id, double epsilon, void* out, int64_t N, mt_stream stream);
int mt_norm_act_bwd(int dtype, const void* x, const void* grad_out, int dim, int num_channels,
                    const int32_t* chan_first, const int32_t* chan_dim, int act_id, double epsilon, void* grad_x,
                    int64_t N, mt_stream stream);

/* f4: target normalisers (reference src/matten/data/transform.py:116-133 MeanNormNormalize, :265-279
 * ScalarNormalize).  inverse 0: out = (data - mean) / (norm * scale); inverse 1: out = data * (norm * scale) + mean,
 * each operation rounded separately as the reference's elementwise expressions are.  data/out [N,dim], mean/norm
 * [dim].  The statistics themselves (compute_statistics, :139-216) are column reductions: mt_col_reduce. */
int mt_normalize(int dtype, const void* data, const void* mean, const void* norm, double scale, int inverse,
                 void* out, int64_t N, int dim, mt_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* MATTEN_B200_H */
