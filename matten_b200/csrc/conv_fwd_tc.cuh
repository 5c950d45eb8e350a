// Fused convolution forward, Blackwell-native version (fp32 storage):
//
//   last radial-MLP layer            w[e, c] = sum_k h[e,k] W[k,c] -> tcgen05.mma (bf16 x3 split, fp32 accumulate)
//   accumulators                                                   -> TMEM  (lane = weight column c, column = edge e)
//   gathered sender rows x[src]                                    -> TMA tile::gather4 (4 rows per instruction)
//   uvu Clebsch-Gordan contraction + per-receiver sum              -> FP32 FMA pipes (FFMA2: two edges per instruction),
//                                                                     operands in shared memory, per-node sums in
//                                                                     registers (CSR order, no atomics)
//
// Same contract as conv_fwd.cuh (reference src/matten/nn/utils.py:260-263 + src/matten/nn/conv.py:113-120): the
// per-edge tensor-product weights [E, weight_numel] and the messages [E, D_mid] never leave the SM.
//
// Kernels:
//  (0) once per batch (mt_conv_layout_prepare; or at every call when the caller passes no layout):
//      tc_pad_degree / scan / tc_pad_layout_kernel: the receiver-sorted edge list in PADDED column order -- every
//      node's edges padded to a multiple of 4 columns (pad columns repeat the node's last edge and get zero weights):
//      per column the original edge id and the sender row.  With this layout every chunk of the fused kernel is ONE
//      contiguous column range.  tc_ypairs_kernel: the edges' spherical harmonics as pair-interleaved padded rows.
//  (1) tc_edge_hidden_fast_kernel (MLP shape <= 8 -> 32 -> 32, silu; tc_edge_hidden_kernel otherwise): the small
//      hidden layers of the radial MLP per column, written as three bf16 planes (hi / mid / lo) in the K-major
//      core-matrix layout the MMA wants (192 bytes per column).
//      (Round 2 also built this stage INTO the fused kernel, on dedicated warps: correct, but slower -- a lone warp
//      per scheduler runs such code at ~10 cycles per instruction and the h planes of the next chunk sat on the
//      critical path; measurements in DESIGN.md.)
//  (2) conv_fwd_tc_kernel: 1 CTA per SM, persistent over a contiguous node range (balanced by edge count), 20 warps:
//        warp 0      builds node-aligned chunks (<= NE columns) and issues the copies of the chunk: one 3D TMA tile
//                    load of the twelve h-plane segments and one bulk copy of the sh pair rows;
//        warp 1      one thread issues the tcgen05.mma's of the chunk: D[t] (128 x NE, TMEM) = A[t] (128 rows of W^T,
//                    K = 32) x B^T (NE columns), 6 significant products of the 3 x 3 bf16 split (~2^-24);
//        warp 2      TMA gathers of the sender rows, 4 rows per instruction (warp 3 takes the odd groups for one-tile
//                    parts, whose chunks are 256 columns; it idles otherwise);
//        warps 4..19 consumers.  Warp w reads TMEM lanes 32 (w % 4) .. .  Work units (bundle instance, node) are
//                    handed out dynamically per quarter.  A bundle instance (matten_b200/tcplan.py) is a group of
//                    input channels x a compile-time list of paths that share the loads of x[u, :] and Y
//                    (generated/cg_bundles.cuh):
//                      mode L: lane == channel (32 channels), the warp walks the node's edge pairs;
//                      mode P: 8 / 4 / 2 channels x edge phases through the tcgen05.ld.16x256b fragment
//                              (thread 4 r + ph: TMEM rows r and r + 8, column pair ph of 4).
//      Double buffered TMEM accumulators and x / Y staging; mbarriers: full[b] (copy bytes + tcgen05.commit),
//      empty[b] (consumers), go[b] (gather warps), bready / bfree (h planes landed / consumed by the MMAs).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "generated/cg_bundles.cuh"

namespace mt {

constexpr int kTcK = 32;              // padded size of the last hidden layer == MMA K total
constexpr int kTcProducerWarps = 4;   // warp 0: chunks + plane / sh copies, warp 1: MMA issue, warps 2 and 3: TMA gathers (even / odd groups)
constexpr int kTcConsumerWarps = 16;  // a multiple of 4: warp w reads TMEM quarter w % 4
constexpr int kTcThreads = 32 * (kTcProducerWarps + kTcConsumerWarps);
constexpr int kTcMaxTiles = 4;        // M tiles of 128 rows per part
constexpr int kTcMaxBI = 64;          // bundle instances per part
constexpr int kTcMaxNodes = 32;       // receiver nodes per chunk
constexpr int kTcMaxParts = 4;

// columns (padded edges) per chunk == MMA N: 2 stages x MT tiles x NE columns must fit the 512 TMEM columns
__host__ __device__ constexpr int tc_chunk_cols(int MT) { return MT <= 1 ? 256 : (MT == 2 ? 128 : (MT == 3 ? 80 : 64)); }

struct TcPartParams {
  int num_tiles;             // MT
  int a_rows;                // rows of the A operand kept in shared memory (a multiple of 32, > the last used row)
  int num_bi;
  int x_lo, x_cols;          // gathered window of the x row (floats): TMA column coordinate and box width
  int ne;                    // chunk columns
  int cta_first, cta_count;  // CTAs [cta_first, cta_first + cta_count) run this part
  int q_count[4];
  const int32_t* row_wcol;   // [MT*128] weight column of every A row (-1: zero row)
  const int32_t* bi_hdr;     // [num_bi][8] {bundle id, mode, nch, mask, quarter, slot0, slot1, slot2}
  const int32_t* bi_lane;    // [num_bi][32][4] per lane {x offset in the window, out offset of path 0 / 1 / 2 (-1: none)}
  const int32_t* q_list;     // [4][kTcMaxBI] bundle instances per quarter (heavy first)
};

struct ConvTcParams {
  int x_dim, y_dim, y_lmax, out_dim;
  int nl;
  int sizes[MT_MAX_MLP_LAYERS + 1];
  int act;
  float act_cst;
  const float* w[MT_MAX_MLP_LAYERS];
  const float* emb;
  const int32_t* rowptr;
  const int32_t* perm;
  const int32_t* src;
  // per-batch edge layout (kernels (0)), except hplanes (workspace, kernel (1))
  int32_t* rowptr_pad;        // [N+1] first padded column of every node (multiples of 4); [N] = number of columns
  int32_t* orig_pad;          // [cols] original edge id of the column (pad column: -1 - id of the node's last edge)
  int32_t* src_pad;           // [cols] sender row of the column
  __nv_bfloat16* hplanes;     // [3][4][cols_max][8] bf16: plane, k-group, column, k % 8
  float* ypairs;              // [cols_max / 2][2 * y_pad]: pair-interleaved padded sh rows
  int64_t cols_max;           // allocated columns (E + 3 N rounded up to 4)
  float avg;
  const float* num_neigh;
  float* out;
  int64_t N, E;
  int num_parts;
  TcPartParams part[kTcMaxParts];
  long long* dbg;  // optional phase-timing buffer (mt_conv_set_debug_buffer): [warp][8] clock64 sums of CTA 0
};

struct alignas(64) TcMaps {
  CUtensorMap m[kTcMaxParts];  // x as a 2D tensor [N][x_dim], box {x_cols, 1}: one per part (its column window)
  CUtensorMap h[kTcMaxParts];  // h planes as a 3D tensor [12][cols_max][16 bytes], box {16, NE, 12}: one per part (its NE)
};

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Bounded wait: a protocol bug (or a faulted copy) must end in a trap with a message, never in a hang.
__device__ __noinline__ void mbar_timeout(int id, uint32_t parity) {
  printf("[matten_b200] mbarrier wait timed out: barrier %d parity %u block %d warp %d\n", id, parity, (int)blockIdx.x,
         (int)(threadIdx.x >> 5));
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int id = 0) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
  long long t0 = 0;
  uint32_t spins = 0;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(2000u)  // suspend-time hint (ns): the warp sleeps in hardware instead of polling
        : "memory");
    if (!done) {
      // back off: the issue arbiter favours high warp ids, a waiter that polls at full rate starves the working
      // warps of its scheduler (measured: 20 cycles per instruction for the producers with polling consumers)
      __nanosleep(spins < 8 ? 40 : 200);
      if ((++spins & 1023u) == 0) {  // ~2 s: far beyond any legitimate wait in this kernel
        const long long now = clock64();
        if (t0 == 0) t0 = now;
        else if (now - t0 > 4000000000ll) mbar_timeout(id, parity);
      }
    }
  } while (!done);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, bf16 inputs, fp32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// tcgen05.ld is asynchronous: the destination registers are valid only after tcgen05.wait::ld.  The wait (and the
// empty "touch" statements for further register groups) take the registers as read-write operands so the compiler
// cannot move a use above it.  (Scalars, not arrays: arrays passed through asm operands end up in local memory.)
struct W4 {
  uint32_t a, b, c, d;
};
__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, W4& r) {  // lane == TMEM lane, 4 consecutive columns
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.a), "=r"(r.b), "=r"(r.c), "=r"(r.d)
               : "r"(taddr));
}
// 16 lanes x 8 columns: thread 4 r + ph gets (lane r: columns 2 ph, 2 ph + 1; lane r + 8: the same columns)
__device__ __forceinline__ void tmem_ld_16x256b(uint32_t taddr, W4& r) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.a), "=r"(r.b), "=r"(r.c), "=r"(r.d)
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(W4& r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r.a), "+r"(r.b), "+r"(r.c), "+r"(r.d));
}
__device__ __forceinline__ void tmem_ld_touch(W4& r) {  // no instruction: orders uses of r after the preceding wait
  asm volatile("" : "+r"(r.a), "+r"(r.b), "+r"(r.c), "+r"(r.d));
}

// TMA tile::gather4: rows r0..r3 of the 2D tensor, columns [col, col + box) -> 4 consecutive rows of shared memory
__device__ __forceinline__ void tma_gather4(void* dst_smem, const CUtensorMap* map, int col, int r0, int r1, int r2, int r3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes.cta_group::1 "
      "[%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(smem_u32(dst_smem)),
      "l"(map), "r"(col), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(smem_u32(bar))
      : "memory");
}

// TMA tile load of a 3D box (the 12 h-plane segments of a chunk in ONE instruction; out-of-range columns are zero
// filled and still counted in the transaction bytes)
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst_smem)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}

// bulk asynchronous copy global -> shared (the non-tensor TMA path); completes bytes on an mbarrier.
// size and both addresses are multiples of 16 bytes.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// K-major, no-swizzle ("interleave") shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, sm100):
//   element (row r, k) of a [rows x 16] bf16 K-step lives at
//   start + (r/8)*SBO + (k/8)*LBO + (r%8)*16 + (k%8)*2   bytes
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t start_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((start_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version 1 (Blackwell)
  return d;                // base_offset 0, lbo_mode 0, layout_type 0 (SWIZZLE_NONE)
}
// cute::UMMA::InstrDescriptor for kind::f16: BF16 x BF16 -> F32, both K-major
__device__ __forceinline__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void split_bf16x3(float v, __nv_bfloat16& hi, __nv_bfloat16& mi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  const float r1 = v - __bfloat162float(hi);
  mi = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(mi);
  lo = __float2bfloat16_rn(r2);
}

// phase timing of CTA 0 (only when a debug buffer is set): TACC(i) adds the cycles since the last stamp to slot i
#define MT_TC_TIMER() const bool _tm = (p.dbg != nullptr) && blockIdx.x == 0; unsigned _tl = _tm ? (unsigned)clock() : 0u; unsigned _ta[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define MT_TACC(i) do { if (_tm) { const unsigned _n = (unsigned)clock(); _ta[i] += (_n - _tl) >> 4; _tl = _n; } } while (0)
#define MT_TC_TIMER_FLUSH() do { if (_tm && lane == 0) { for (int _i = 0; _i < 8; ++_i) p.dbg[warp * 8 + _i] = (long long)_ta[_i] << 4; } } while (0)

struct __align__(16) TcMeta {
  int nnodes;  // -1: terminate
  int ncols;   // used (padded) columns; 0: only nodes without edges
  int continues;  // 1: the first node of the chunk continues a node split over chunks
  int pc0;        // first padded column of the chunk
  int node_id[kTcMaxNodes];
  float inv_den[kTcMaxNodes];        // 1 / sqrt(avg_num_neighbors) or 1 / sqrt(num_neigh[node])
  short cb[kTcMaxNodes];             // first column of the node (multiple of 4)
  short ngrp[kTcMaxNodes];           // padded edge count / 4
  unsigned char first[kTcMaxNodes];  // 1: this chunk holds the node's first edges (plain store), 0: accumulate
};

// shared-memory carve-up (bytes); every sub-buffer starts at a multiple of 128
struct TcSmemLayout {
  size_t a_off, a_plane;  // 3 planes of [a_rows x 32] bf16 (the MMAs of the last tile read past a_rows into the next
                          // plane / the B planes: rows nobody uses)
  size_t b_off, b_plane;  // 3 planes of [NE x 32] bf16
  size_t x_off, x_buf;    // 2 buffers [NE][x_cols] fp32
  size_t y_off, y_buf;    // 2 buffers [NE/2][2 * y_pad] fp32 (pair-interleaved sh rows)
  size_t meta_off;        // 2 TcMeta
  size_t lane_off;        // [num_bi][32] int4
  size_t hdr_off;         // [num_bi][8] int
  size_t qlist_off;       // [4][kTcMaxBI] uint8
  size_t total;
};
__host__ __device__ inline size_t tc_align(size_t v, size_t a = 128) { return (v + a - 1) & ~(a - 1); }
__host__ __device__ inline int tc_pad8(int v) { return (v + 7) & ~7; }
__host__ __device__ inline TcSmemLayout tc_smem_layout(int a_rows, int x_cols, int y_pad, int num_bi, int NE) {
  TcSmemLayout L;
  size_t o = 0;
  L.a_off = o;
  L.a_plane = (size_t)a_rows * kTcK * 2;
  o += 3 * L.a_plane;
  L.b_off = o;
  L.b_plane = (size_t)NE * kTcK * 2;
  o = tc_align(o + 3 * L.b_plane);
  L.x_off = o;
  L.x_buf = tc_align((size_t)NE * x_cols * 4);
  o += 2 * L.x_buf;
  L.y_off = o;
  L.y_buf = tc_align((size_t)(NE / 2) * 2 * y_pad * 4);
  o += 2 * L.y_buf;
  L.meta_off = o;
  o = tc_align(o + 2 * tc_align(sizeof(TcMeta), 16));
  L.lane_off = o;
  o += (size_t)num_bi * 32 * 16;
  L.hdr_off = o;
  o += (size_t)num_bi * 32;
  L.qlist_off = o;
  o = tc_align(o + 4 * kTcMaxBI);
  L.total = o;
  return L;
}

// =====================================================================================================
// consumer units
// =====================================================================================================
struct TcUnit {
  uint32_t tstage;    // TMEM address of the stage: base + b * MT * NE columns (lane field 0)
  int quarter;        // TMEM lanes 32 * quarter ..
  int ne;             // chunk columns
  int slot[3];        // per path: 2 * tile + half
  unsigned mask;      // active paths
  int nch;            // mode P: channels per row block (8 / 4 / 2)
  const float* xs;    // staged x rows of the chunk [NE][xstride]
  int xstride;
  const float* ys;    // staged pair-interleaved sh rows [NE/2][ystride]
  int ystride;        // floats per edge pair
  int cb, ngrp;       // the node's first column and number of 4-column groups
  int4 lt;            // lane table entry {x offset, out offsets}
  float* out;         // the node's output row
  float inv_den;
  bool first;
};

// (TcUnit travels BY VALUE through force-inlined functions: a unit kept in local memory costs an L2 round trip per
//  field access, the 227 KB shared-memory carve-out leaves almost no L1)
template <class B>
__device__ __forceinline__ void tc_store(const f2* __restrict__ acc, const TcUnit u, unsigned mask) {
  const int oo[3] = {u.lt.y, u.lt.z, u.lt.w};
#pragma unroll
  for (int p = 0; p < B::NP; ++p) {
    if (!((mask >> p) & 1u) || oo[p] < 0) continue;
    float* o = u.out + oo[p];
#pragma unroll
    for (int m = 0; m < B::path_d3(p); ++m) {
      const int i = B::path_acc(p) + m;
      const float v = (acc[i].v.x + acc[i].v.y) * (B::scale(i) * u.inv_den);
      const float prev = u.first ? 0.f : o[m];  // `first` is warp-uniform; one store either way (compact code)
      o[m] = prev + v;
    }
  }
}

template <class B>
__device__ __forceinline__ void tc_load_xy(const TcUnit u, int col, f2* __restrict__ x2, f2* __restrict__ y2) {
  const float* xr = u.xs + (size_t)col * u.xstride + u.lt.x;
#pragma unroll
  for (int m = 0; m < B::D1; ++m) x2[m] = f2(xr[m], xr[u.xstride + m]);
  const float4* yr = reinterpret_cast<const float4*>(u.ys + (size_t)(col >> 1) * u.ystride + 2 * B::Y_LO);
#pragma unroll
  for (int i = 0; i < B::Y_CNT / 2; ++i) {
    const float4 v = yr[i];
    y2[2 * i] = f2(v.x, v.y);
    y2[2 * i + 1] = f2(v.z, v.w);
  }
}

// the same loads through running pointers (mode L walks consecutive pairs: additive addressing only)
template <class B>
__device__ __forceinline__ void tc_load_xy_ptr(const float* __restrict__ xr, int xstride, const float* __restrict__ yp,
                                               f2* __restrict__ x2, f2* __restrict__ y2) {
#pragma unroll
  for (int m = 0; m < B::D1; ++m) x2[m] = f2(xr[m], xr[xstride + m]);
  const float4* yr = reinterpret_cast<const float4*>(yp);
#pragma unroll
  for (int i = 0; i < B::Y_CNT / 2; ++i) {
    const float4 v = yr[i];
    y2[2 * i] = f2(v.x, v.y);
    y2[2 * i + 1] = f2(v.z, v.w);
  }
}

// Both unit loops are kept SMALL on purpose (one edge pair per iteration, no per-path branches when every path of the
// bundle exists): five warps per scheduler run five different instruction streams, and a loop body that does not stay
// in the instruction cache stalls on every 128-byte line (ncu: `no_instruction` was the top stall of the unrolled form).
struct W2 {
  uint32_t a, b;
};
__device__ __forceinline__ void tmem_ld_x2(uint32_t taddr, W2& r) {  // lane == TMEM lane, 2 consecutive columns
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r.a), "=r"(r.b) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait2(W2& r) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(r.a), "+r"(r.b));
}
__device__ __forceinline__ void tmem_ld_touch2(W2& r) { asm volatile("" : "+r"(r.a), "+r"(r.b)); }

// mode L: lane == channel; every lane walks all edge pairs of the node, two edges per FFMA2
template <class B, bool FULL>
__device__ __forceinline__ void tc_unit_L(const TcUnit u) {
  constexpr unsigned kAll = (1u << B::NP) - 1u;
  const unsigned mask = FULL ? kAll : u.mask;
  f2 acc[B::NACC];
#pragma unroll
  for (int i = 0; i < B::NACC; ++i) acc[i] = f2(0.f, 0.f);
  const uint32_t tq = u.tstage + ((uint32_t)(32 * u.quarter) << 16) + (uint32_t)u.cb;
  uint32_t ta[B::NP];
#pragma unroll
  for (int p = 0; p < B::NP; ++p) ta[p] = tq + (uint32_t)((u.slot[p] >> 1) * u.ne);
  W2 wc[B::NP], wn[B::NP];
#pragma unroll
  for (int p = 0; p < B::NP; ++p) {
    wc[p].a = wc[p].b = 0u;
    wn[p] = wc[p];
  }
  const int npairs = 2 * u.ngrp;
  if (npairs > 0) {
#pragma unroll
    for (int p = 0; p < B::NP; ++p)
      if ((mask >> p) & 1u) tmem_ld_x2(ta[p], wc[p]);
    tmem_ld_wait2(wc[0]);
#pragma unroll
    for (int p = 1; p < B::NP; ++p) tmem_ld_touch2(wc[p]);
  }
  const float* xr = u.xs + (size_t)u.cb * u.xstride + u.lt.x;                       // += 2 rows per pair
  const float* yp = u.ys + (size_t)(u.cb >> 1) * u.ystride + 2 * B::Y_LO;           // += 1 pair row per pair
  const int xstep = 2 * u.xstride;
  uint32_t tnext = 2u;
#pragma unroll 1
  for (int g = 0; g < npairs; ++g) {
    const bool more = g + 1 < npairs;
    if (more) {
#pragma unroll
      for (int p = 0; p < B::NP; ++p)
        if ((mask >> p) & 1u) tmem_ld_x2(ta[p] + tnext, wn[p]);  // prefetch the next pair's weights
      tnext += 2u;
    }
    f2 x2[B::D1], y2[B::Y_CNT], w2[B::NP];
    tc_load_xy_ptr<B>(xr, u.xstride, yp, x2, y2);
    xr += xstep;
    yp += u.ystride;
#pragma unroll
    for (int p = 0; p < B::NP; ++p) w2[p] = f2(__uint_as_float(wc[p].a), __uint_as_float(wc[p].b));
    B::template edge<f2>(x2, y2, w2, acc, mask);
    if (more) {
      tmem_ld_wait2(wn[0]);
#pragma unroll
      for (int p = 1; p < B::NP; ++p) tmem_ld_touch2(wn[p]);
#pragma unroll
      for (int p = 0; p < B::NP; ++p) wc[p] = wn[p];
    }
  }
  tc_store<B>(acc, u, mask);
}

// mode P: thread 4 r + ph: channel r % nch, edge pairs ph + 4 (r / nch) of every block of 32 / nch pairs
template <class B, bool FULL>
__device__ __forceinline__ void tc_unit_P(const TcUnit u, int lane) {
  constexpr int NPAIR = (B::NP + 1) / 2;
  constexpr unsigned kAll = (1u << B::NP) - 1u;
  const unsigned mask = FULL ? kAll : u.mask;
  f2 acc[B::NACC];
#pragma unroll
  for (int i = 0; i < B::NACC; ++i) acc[i] = f2(0.f, 0.f);
  const int r8 = lane >> 2, ph = lane & 3;
  const int lg = (u.nch == 8) ? 3 : (u.nch == 4 ? 2 : 1);
  const int sub = r8 >> lg, dup = 8 >> lg;
  const int block = 8 * dup, ncols = 4 * u.ngrp;
  uint32_t ta[NPAIR];
#pragma unroll
  for (int j = 0; j < NPAIR; ++j) {
    const int s = u.slot[2 * j];  // both paths of a pair share the half slot
    ta[j] = u.tstage + ((uint32_t)(32 * u.quarter + 16 * (s & 1)) << 16) + (uint32_t)((s >> 1) * u.ne);
  }
#pragma unroll 1
  for (int start = u.cb; start < u.cb + ncols; start += block) {
    const int cstart = min(start, u.ne - block);  // keep the TMEM read inside the stage
    W4 wsel[NPAIR];
#pragma unroll
    for (int j = 0; j < NPAIR; ++j) {
      wsel[j].a = wsel[j].b = wsel[j].c = wsel[j].d = 0u;
      if (!((mask >> (2 * j)) & 3u)) continue;  // neither path of the pair exists (warp uniform)
#pragma unroll 1
      for (int d = 0; d < dup; ++d) {
        W4 t;
        tmem_ld_16x256b(ta[j] + (uint32_t)(cstart + 8 * d), t);
        tmem_ld_wait(t);
        if (d == sub) wsel[j] = t;
      }
    }
    const int mycol = cstart + 8 * sub + 2 * ph;
    const bool active = mycol >= start && mycol < u.cb + ncols;
    f2 x2[B::D1], y2[B::Y_CNT], w2[B::NP];
    tc_load_xy<B>(u, active ? mycol : u.cb, x2, y2);
#pragma unroll
    for (int p = 0; p < B::NP; ++p) {
      const W4& t = wsel[p >> 1];
      const float w0 = __uint_as_float((p & 1) ? t.c : t.a), w1 = __uint_as_float((p & 1) ? t.d : t.b);
      w2[p] = active ? f2(w0, w1) : f2(0.f, 0.f);
    }
    B::template edge<f2>(x2, y2, w2, acc, mask);
    __syncwarp();
  }
  // fixed-order butterfly over the edge phases (lane bits 0-1) and the duplicate row blocks (lane bits 2+lg ..)
#pragma unroll
  for (int i = 0; i < B::NACC; ++i) {
    float s = acc[i].v.x + acc[i].v.y;
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    for (int o = 4 << lg; o < 32; o <<= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    acc[i] = f2(s, 0.f);
  }
  tc_store<B>(acc, u, mask);
}

template <int ID>
__device__ __forceinline__ void tc_unit_dispatch(const TcUnit u, int mode, int lane) {
  using B = Bundle<ID>;
  const bool full = u.mask == (1u << B::NP) - 1u;
  if (mode == 0) {
    if (full) tc_unit_L<B, true>(u);
    else tc_unit_L<B, false>(u);
  } else {
    if (full) tc_unit_P<B, true>(u, lane);
    else tc_unit_P<B, false>(u, lane);
  }
}

// =====================================================================================================
// preparation kernels: padded column order, hidden layers of the radial MLP, sh pair rows
// =====================================================================================================
// sigmoid through the special-function unit: ex2.approx (2 ulp) and rcp.approx (1 ulp); relative error ~3e-7
__device__ __forceinline__ float tc_fast_sigmoid(float v) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * v));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return r;
}
// hi / mid / lo bf16 planes of 8 floats (v = hi + mid + lo to ~2^-24), packed conversions (two values per F2FP)
__device__ __forceinline__ void tc_split8(const float (&v)[8], uint4& hi, uint4& mi, uint4& lo) {
  uint32_t H[4], M[4], Lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float a = v[2 * i], b = v[2 * i + 1];
    const __nv_bfloat162 h2 = __floats2bfloat162_rn(a, b);
    const uint32_t hb = *reinterpret_cast<const uint32_t*>(&h2);
    const float ra = a - __uint_as_float(hb << 16), rb = b - __uint_as_float(hb & 0xffff0000u);
    const __nv_bfloat162 m2 = __floats2bfloat162_rn(ra, rb);
    const uint32_t mb = *reinterpret_cast<const uint32_t*>(&m2);
    const float sa = ra - __uint_as_float(mb << 16), sb = rb - __uint_as_float(mb & 0xffff0000u);
    const __nv_bfloat162 l2 = __floats2bfloat162_rn(sa, sb);
    H[i] = hb;
    M[i] = mb;
    Lo[i] = *reinterpret_cast<const uint32_t*>(&l2);
  }
  hi = make_uint4(H[0], H[1], H[2], H[3]);
  mi = make_uint4(M[0], M[1], M[2], M[3]);
  lo = make_uint4(Lo[0], Lo[1], Lo[2], Lo[3]);
}

// padded degrees (multiples of 4), to be scanned into rowptr_pad
__global__ void __launch_bounds__(256) tc_pad_degree_kernel(const int32_t* __restrict__ rowptr, int64_t N,
                                                            int32_t* __restrict__ degp) {
  const int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (n < N) degp[n] = (rowptr[n + 1] - rowptr[n] + 3) & ~3;
  if (n == N) degp[n] = 0;
}

// one warp per node: the node's padded columns
__global__ void __launch_bounds__(256) tc_pad_layout_kernel(const int32_t* __restrict__ rowptr,
                                                            const int32_t* __restrict__ rowptr_pad,
                                                            const int32_t* __restrict__ perm, const int32_t* __restrict__ src,
                                                            int64_t N, int32_t* __restrict__ orig_pad,
                                                            int32_t* __restrict__ src_pad) {
  const int lane = threadIdx.x & 31;
  for (int64_t n = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; n < N; n += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int r0 = rowptr[n], deg = rowptr[n + 1] - r0;
    const int c0 = rowptr_pad[n], degp = rowptr_pad[n + 1] - c0;
    for (int t = lane; t < degp; t += 32) {
      const int e = r0 + (t < deg ? t : deg - 1);  // pad columns repeat the node's last edge
      const int o = perm[e];
      orig_pad[c0 + t] = (t < deg) ? o : (-1 - o);
      src_pad[c0 + t] = src[e];
    }
  }
}

// hidden layers: four lanes per column (lane q4 produces outputs 8 q4 .. 8 q4 + 7), 8 columns per warp pass; layer
// inputs / outputs are exchanged through a shared-memory row per column (stride 33: conflict free)
constexpr int kHidThreads = 256;
__global__ void __launch_bounds__(kHidThreads) tc_edge_hidden_kernel(const ConvTcParams p) {
  __shared__ __align__(16) float sW[2 * kTcK * kTcK];
  __shared__ float sV[(kHidThreads / 32) * 8 * 33];
  const int nh = p.nl - 1;
  for (int li = 0; li < nh; ++li) {
    const int fi = p.sizes[li], fo = p.sizes[li + 1];
    const float s = rsqrtf((float)fi);
    for (int t = threadIdx.x; t < kTcK * kTcK; t += kHidThreads) {
      const int k = t >> 5, j = t & 31;
      sW[li * kTcK * kTcK + t] = (k < fi && j < fo) ? p.w[li][(size_t)k * fo + j] * s : 0.f;
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q4 = lane & 3, cl = lane >> 2;
  const int in0 = p.sizes[0];
  float* vrow = sV + (warp * 8 + cl) * 33;
  const int64_t cols = p.rowptr_pad[p.N];
  uint4* planes = reinterpret_cast<uint4*>(p.hplanes);
  const int64_t wpb = kHidThreads / 32;
  for (int64_t c0 = (blockIdx.x * wpb + warp) * 8; c0 < cols; c0 += (int64_t)gridDim.x * wpb * 8) {
    const int64_t c = c0 + cl;  // cols is a multiple of 4: a block of 8 may end half way
    const bool in = c < cols;
    const int oe = in ? p.orig_pad[c] : 0;
    const bool real = in && oe >= 0;
    const int64_t orig = oe >= 0 ? oe : (-1 - oe);
    const float* er = p.emb + orig * in0;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = 8 * q4 + i;
      vrow[idx] = (real && idx < in0) ? er[idx] : 0.f;
    }
    __syncwarp();
#pragma unroll 1
    for (int li = 0; li < nh; ++li) {
      const int K = p.sizes[li], fo = p.sizes[li + 1];
      const float* W = sW + li * kTcK * kTcK + 8 * q4;
      float2 a[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = make_float2(0.f, 0.f);
#pragma unroll 8
      for (int kk = 0; kk < K; ++kk) {
        const float hk = vrow[kk];
        const float4* wr = reinterpret_cast<const float4*>(W + kk * kTcK);
        const float4 w0 = wr[0], w1 = wr[1];
        fma_pair(hk, w0.x, w0.y, a[0]);
        fma_pair(hk, w0.z, w0.w, a[1]);
        fma_pair(hk, w1.x, w1.y, a[2]);
        fma_pair(hk, w1.z, w1.w, a[3]);
      }
      __syncwarp();  // all four lanes of the column have read the inputs
      float o8[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        o8[2 * i] = a[i].x;
        o8[2 * i + 1] = a[i].y;
      }
      if (p.act == MT_ACT_SILU) {  // the eight chains are independent: the special-function unit pipelines them
#pragma unroll
        for (int i = 0; i < 8; ++i) o8[i] = o8[i] * tc_fast_sigmoid(o8[i]);
      } else {
#pragma unroll 1
        for (int i = 0; i < 8; ++i) o8[i] = apply_act<float>(p.act, o8[i]);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) vrow[8 * q4 + i] = (8 * q4 + i < fo) ? o8[i] * p.act_cst : 0.f;
      __syncwarp();
    }
    if (in) {
      float h8[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) h8[i] = real ? vrow[8 * q4 + i] : 0.f;  // pad column: zero weights
      uint4 hi, mi, lo;
      tc_split8(h8, hi, mi, lo);
      planes[(size_t)(0 * 4 + q4) * p.cols_max + c] = hi;  // k-group q4 of the column
      planes[(size_t)(1 * 4 + q4) * p.cols_max + c] = mi;
      planes[(size_t)(2 * 4 + q4) * p.cols_max + c] = lo;
    }
  }
}

// sh rows -> pair-interleaved padded rows (degree-l block at position sh_pad_pos(l)), one lane per column: the only
// writer of ypairs
__global__ void __launch_bounds__(256) tc_ypairs_kernel(const float* __restrict__ sh, const int32_t* __restrict__ rowptr_pad,
                                                        const int32_t* __restrict__ orig_pad, int64_t N, int ylmax,
                                                        float* __restrict__ ypairs) {
  const int yn = (ylmax + 1) * (ylmax + 1);
  const int ystride = 2 * sh_pad_len(ylmax);
  const int64_t cols = rowptr_pad[N];
  for (int64_t c = blockIdx.x * 256ll + threadIdx.x; c < cols; c += (int64_t)gridDim.x * 256) {
    const int oe = orig_pad[c];
    const int64_t orig = oe >= 0 ? oe : (-1 - oe);
    const float* __restrict__ yr = sh + orig * yn;
    float* yo = ypairs + (c >> 1) * ystride + (c & 1);
#pragma unroll
    for (int l = 0; l <= MT_LMAX; ++l) {
      if (l <= ylmax) {
#pragma unroll
        for (int k = 0; k < 2 * l + 1; ++k) yo[2 * (sh_pad_pos(l) + k)] = yr[l * l + k];
      }
    }
  }
}

// The same stage for the MLP shape every matten config uses (n_rad <= 8 -> 32 -> 32 -> W, silu): lane == column, all
// 32 hidden outputs of the column in registers, weights by warp-wide broadcast LDS.128.  Per input channel a lane
// issues 8 LDS.128 and 16 FFMA2 and nothing else (the generic kernel above spends 40 % of its instructions on
// predicates, index arithmetic and the shared-memory exchange between its four lanes per column: ncu r2_step_full).
__global__ void __launch_bounds__(256, 3) tc_edge_hidden_fast_kernel(const ConvTcParams p) {
  __shared__ __align__(16) float sW0[8 * kTcK];
  __shared__ __align__(16) float sW1[kTcK * kTcK];
  const int in0 = p.sizes[0];
  {
    const float s0 = rsqrtf((float)in0), s1 = rsqrtf((float)kTcK);
    for (int t = threadIdx.x; t < 8 * kTcK; t += 256) sW0[t] = (t >> 5) < in0 ? p.w[0][t] * s0 : 0.f;
    for (int t = threadIdx.x; t < kTcK * kTcK; t += 256) sW1[t] = p.w[1][t] * s1;
  }
  __syncthreads();
  const uint32_t cols = p.rowptr_pad[p.N];  // < 2^31 (E + 3 N < 2^31): 32-bit column indices save registers
  uint4* planes = reinterpret_cast<uint4*>(p.hplanes);
  const float cst = p.act_cst;
  const bool emb_vec = in0 == 8 && (reinterpret_cast<uintptr_t>(p.emb) & 15) == 0;
  for (uint32_t c = blockIdx.x * 256 + threadIdx.x; c < cols; c += gridDim.x * 256) {
    const int oe = p.orig_pad[c];
    const bool real = oe >= 0;
    const int64_t orig = real ? oe : (-1 - oe);
    float h0[8];
    if (emb_vec) {
      const float4* er = reinterpret_cast<const float4*>(p.emb + orig * 8);
      const float4 a = er[0], b = er[1];
      h0[0] = a.x; h0[1] = a.y; h0[2] = a.z; h0[3] = a.w;
      h0[4] = b.x; h0[5] = b.y; h0[6] = b.z; h0[7] = b.w;
    } else {
      const float* er = p.emb + orig * in0;
#pragma unroll
      for (int i = 0; i < 8; ++i) h0[i] = i < in0 ? er[i] : 0.f;
    }
    float2 acc[16];
    float h1[kTcK];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float4* wr = reinterpret_cast<const float4*>(sW0 + k * kTcK);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 w = wr[j];
        fma_pair(h0[k], w.x, w.y, acc[2 * j]);
        fma_pair(h0[k], w.z, w.w, acc[2 * j + 1]);
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      h1[2 * i] = acc[i].x * tc_fast_sigmoid(acc[i].x) * cst;
      h1[2 * i + 1] = acc[i].y * tc_fast_sigmoid(acc[i].y) * cst;
      acc[i] = make_float2(0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < kTcK; ++k) {
      const float4* wr = reinterpret_cast<const float4*>(sW1 + k * kTcK);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 w = wr[j];
        fma_pair(h1[k], w.x, w.y, acc[2 * j]);
        fma_pair(h1[k], w.z, w.w, acc[2 * j + 1]);
      }
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      float h8[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = acc[4 * g + i].x, b = acc[4 * g + i].y;
        h8[2 * i] = real ? a * tc_fast_sigmoid(a) * cst : 0.f;  // pad column: zero weights
        h8[2 * i + 1] = real ? b * tc_fast_sigmoid(b) * cst : 0.f;
      }
      uint4 hi, mi, lo;
      tc_split8(h8, hi, mi, lo);
      planes[(size_t)(0 * 4 + g) * p.cols_max + c] = hi;  // k-group g of the column
      planes[(size_t)(1 * 4 + g) * p.cols_max + c] = mi;
      planes[(size_t)(2 * 4 + g) * p.cols_max + c] = lo;
    }
  }
}

// =====================================================================================================
// the kernel.  LMAXK: largest degree of the bundles compiled in (2: l <= 2 layers, 4: everything)
// =====================================================================================================
template <int LMAXK>
__global__ void __launch_bounds__(kTcThreads, 1) conv_fwd_tc_kernel(const __grid_constant__ ConvTcParams p,
                                                                   const __grid_constant__ TcMaps maps) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t bar_full[2], bar_empty[2], bar_go[2], bar_bready, bar_bfree;
  __shared__ uint32_t s_tmem_base;
  __shared__ int s_cnt[2][4];
  __shared__ int s_mma_b;  // buffer of the chunk handed to the MMA warp (-1: terminate)

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // which part does this CTA run, and which share of the node range
  int part_id = 0;
#pragma unroll
  for (int i = 1; i < kTcMaxParts; ++i)
    if (i < p.num_parts && (int)blockIdx.x >= p.part[i].cta_first) part_id = i;
  const TcPartParams& P = p.part[part_id];
  const int MT = P.num_tiles, NE = P.ne, a_rows = P.a_rows;
  const int y_pad = sh_pad_len(p.y_lmax);
  const int ystride = 2 * y_pad;
  const TcSmemLayout L = tc_smem_layout(a_rows, P.x_cols, y_pad, P.num_bi, NE);
  unsigned char* sA = smem + L.a_off;
  unsigned char* sB = smem + L.b_off;
  unsigned char* sMeta = smem + L.meta_off;
  constexpr size_t kMetaBytes = (sizeof(TcMeta) + 15) & ~(size_t)15;
  int4* sLane = reinterpret_cast<int4*>(smem + L.lane_off);
  int* sHdr = reinterpret_cast<int*>(smem + L.hdr_off);
  unsigned char* sQ = smem + L.qlist_off;

  // ---------------------------------------------------------------- one-time setup
  if (tid == 0) {
    mbar_init(&bar_full[0], 2);  // producer (copy bytes) + MMA commit
    mbar_init(&bar_full[1], 2);
    mbar_init(&bar_empty[0], kTcConsumerWarps);
    mbar_init(&bar_empty[1], kTcConsumerWarps);
    mbar_init(&bar_go[0], 1);
    mbar_init(&bar_go[1], 1);
    mbar_init(&bar_bready, 1);
    mbar_init(&bar_bfree, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(&s_tmem_base, 512);
  // plan tables -> shared memory (with a ~225 KB carve-out the L1 is a few KB: every global load is an L2 trip)
  for (int t = tid; t < P.num_bi * 32; t += kTcThreads) sLane[t] = reinterpret_cast<const int4*>(P.bi_lane)[t];
  for (int t = tid; t < P.num_bi * 8; t += kTcThreads) sHdr[t] = P.bi_hdr[t];
  for (int t = tid; t < 4 * kTcMaxBI; t += kTcThreads) sQ[t] = (unsigned char)P.q_list[t];
  // staging buffers start zeroed (columns past the chunk's range are never read with non-zero weights, but must be finite)
  {
    uint4* z = reinterpret_cast<uint4*>(smem + L.b_off);
    const int n16 = (int)((L.meta_off - L.b_off) >> 4);  // B planes, x and Y buffers
    for (int t = tid; t < n16; t += kTcThreads) z[t] = make_uint4(0u, 0u, 0u, 0u);
  }
  // A planes: rows of W_last^T (pre-scaled by 1/sqrt(H)) split into bf16 hi/mid/lo, canonical K-major layout
  {
    const int H = p.sizes[p.nl - 1], Wn = p.sizes[p.nl];
    const float* __restrict__ Wl = p.w[p.nl - 1];
    const float s = rsqrtf((float)H);
    for (int t = tid; t < a_rows * 4; t += kTcThreads) {
      const int R = t >> 2, g = t & 3;
      const int wc = P.row_wcol[R];
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = g * 8 + i;
        v[i] = (wc >= 0 && k < H) ? Wl[(size_t)k * Wn + wc] * s : 0.f;
      }
      uint4 hi, mi, lo;
      tc_split8(v, hi, mi, lo);
      const size_t off = (size_t)g * a_rows * 16 + (size_t)R * 16;
      *reinterpret_cast<uint4*>(sA + off) = hi;
      *reinterpret_cast<uint4*>(sA + L.a_plane + off) = mi;
      *reinterpret_cast<uint4*>(sA + 2 * L.a_plane + off) = lo;
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;

  if (warp == 0) {
    // ================================================================ chunk builder + copies
    int64_t n_cur, n_end;
    {
      const int64_t rank = (int64_t)blockIdx.x - P.cta_first, cnt = P.cta_count;
      auto bound = [&](int64_t i) -> int64_t {  // first node whose rowptr >= i*E/cnt
        if (i <= 0) return 0;
        if (i >= cnt) return p.N;
        const int64_t target = (p.E * i) / cnt;
        int64_t lo = 0, hi = p.N;
        while (lo < hi) {
          const int64_t mid = (lo + hi) >> 1;
          if (p.rowptr[mid] < target) lo = mid + 1; else hi = mid;
        }
        return lo;
      };
      if (p.E == 0) {
        n_cur = (p.N * rank) / cnt;
        n_end = (p.N * (rank + 1)) / cnt;
      } else {
        n_cur = bound(rank);
        n_end = bound(rank + 1);
      }
    }
    int c_carry = -1;  // >= 0: the next chunk continues node n_cur at this padded column
    int b_uses = 0;    // chunks that loaded the h planes so far
    const uint32_t xrow_bytes = (uint32_t)P.x_cols * 4, ypair_bytes = (uint32_t)ystride * 4;
    // window of 32 consecutive padded row pointers (lane l: rowptr_pad[w_base + l]) = 31 nodes
    int64_t w_base = n_cur;
    int w_ptr = (w_base + lane <= p.N) ? p.rowptr_pad[w_base + lane] : 0;
    MT_TC_TIMER();  // 0: chunk layout, 1: wait empty, 2: wait bfree, 3: copy issue
    for (int k = 0;; ++k) {
      const int b = k & 1;
      TcMeta& M = *reinterpret_cast<TcMeta*>(sMeta + b * kMetaBytes);
      if (n_cur >= n_end) {
        if (lane == 0) {
          mbar_wait(&bar_empty[b], ((k >> 1) & 1) ^ 1, 10 + b);  // consumers released buffer b
          M.nnodes = -1;
          M.ncols = 0;
          mbar_arrive(&bar_go[b]);  // the gather warp sees the terminator
          if (b_uses > 0) mbar_wait(&bar_bfree, (b_uses - 1) & 1, 20);  // the MMA warp is done with its last chunk
          s_mma_b = -1;
          mbar_arrive(&bar_bready);  // terminator for the MMA warp
          mbar_arrive(&bar_full[b]);
          mbar_arrive(&bar_full[b]);
        }
        break;
      }
      if (n_cur - w_base > 15) {
        w_base = n_cur;
        w_ptr = (w_base + lane <= p.N) ? p.rowptr_pad[w_base + lane] : 0;
      }
      const int off = (int)(n_cur - w_base);
      const int64_t cand = n_cur + lane;  // lane l looks at node n_cur + l
      const bool in_range = cand < n_end && off + lane < 31;
      int c_lo = __shfl_sync(0xffffffffu, w_ptr, (off + lane) & 31);
      const int c_hi = __shfl_sync(0xffffffffu, w_ptr, (off + lane + 1) & 31);
      if (lane == 0 && c_carry >= 0) c_lo = c_carry;
      int degp = in_range ? c_hi - c_lo : 0;  // padded columns of the node (multiple of 4)
      bool split = false;
      if (lane == 0 && degp > NE) {  // node larger than a chunk: take NE columns now, the rest next time
        degp = NE;
        split = true;
      }
      int cum = in_range ? degp : 0x10000;  // inclusive prefix
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, cum, o);
        if (lane >= o) cum += t;
      }
      const unsigned fm = __ballot_sync(0xffffffffu, in_range && cum <= NE);
      int m = (fm == 0xffffffffu) ? 32 : (__ffs(~fm) - 1);  // leading run of nodes that fit
      const bool split0 = __shfl_sync(0xffffffffu, (int)split, 0) != 0;
      if (split0) m = 1;
      const bool mine = lane < m;
      const int cb = cum - degp;
      const float inv_den = mine ? (p.num_neigh ? rsqrtf(p.num_neigh[cand]) : rsqrtf(p.avg)) : 0.f;
      const int ncols = __shfl_sync(0xffffffffu, cum, m - 1);
      const int pc0 = __shfl_sync(0xffffffffu, c_lo, 0);  // first padded column of the chunk
      MT_TACC(0);
      // ---- everything above only read global memory; now wait until the consumers released buffer b
      if (lane == 0) mbar_wait(&bar_empty[b], ((k >> 1) & 1) ^ 1, 10 + b);
      __syncwarp();
      MT_TACC(1);
      if (mine) {
        M.node_id[lane] = (int)cand;
        M.cb[lane] = (short)cb;
        M.ngrp[lane] = (short)(degp >> 2);
        M.first[lane] = (lane == 0 && c_carry >= 0) ? 0 : 1;
        M.inv_den[lane] = inv_den;
      }
      const bool continues = (c_carry >= 0);
      if (lane == 0) {
        M.nnodes = m;
        M.ncols = ncols;
        M.pc0 = pc0;
        s_cnt[b][0] = 0; s_cnt[b][1] = 0; s_cnt[b][2] = 0; s_cnt[b][3] = 0;
        // a chunk that continues a node split over chunks accumulates into its output row: keep the pieces
        // ordered (deterministic sum) by letting the previous chunk drain first
        if (continues && k > 0) mbar_wait(&bar_empty[b ^ 1], ((k - 1) >> 1) & 1, 12);
      }
      __syncwarp();
      if (ncols == 0) {
        if (lane == 0) {
          mbar_arrive(&bar_go[b]);
          mbar_arrive(&bar_full[b]);  // nothing to copy, no MMA: both arrivals from here
          mbar_arrive(&bar_full[b]);
        }
      } else {
        if (lane == 0) {
          mbar_arrive_expect_tx(&bar_full[b], (uint32_t)ncols * xrow_bytes + (uint32_t)(ncols >> 1) * ypair_bytes);
          mbar_arrive(&bar_go[b]);  // warp 2 issues the gathers of the sender rows (a TMA instruction costs ~250 issue
                                    // cycles: 16 gathers + 13 bulk copies on one warp were the critical path)
          if (b_uses > 0) mbar_wait(&bar_bfree, (b_uses - 1) & 1, 21);  // previous MMAs have consumed the h planes
          s_mma_b = b;
          mbar_arrive_expect_tx(&bar_bready, (uint32_t)NE * 16u * 12u);  // the whole box, whatever ncols is
        }
        __syncwarp();
        MT_TACC(2);
        // the chunk is ONE contiguous range of padded columns: 12 plane segments, the sh pair rows, and one TMA gather
        // of 4 sender rows per 4 columns
        // (twelve separate bulk copies cost ~3 k issue cycles per chunk on this warp: each TMA instruction is ~250)
        if (lane == 0) {
          tma_load_3d(sB, &maps.h[part_id], 0, pc0, 0, &bar_bready);
        } else if (lane == 12) {
          bulk_g2s(smem + L.y_off + (size_t)b * L.y_buf, p.ypairs + (size_t)(pc0 >> 1) * ystride,
                   (uint32_t)(ncols >> 1) * ypair_bytes, &bar_full[b]);
        }
        ++b_uses;
        MT_TACC(3);
      }
      // advance
      if (split0) {
        c_carry = pc0 + NE;
        if (c_carry >= __shfl_sync(0xffffffffu, c_hi, 0)) {  // exactly consumed
          c_carry = -1;
          n_cur += 1;
        }
      } else {
        c_carry = -1;
        n_cur += m;
      }
    }
    MT_TC_TIMER_FLUSH();
  } else if (warp == 1) {
    // ================================================================ MMA issuer
    // (two issuing warps, even / odd tiles, were measured: 2-4 % slower -- the MMAs are not what a chunk waits for)
    const uint32_t idesc = make_idesc_bf16(128, NE);
    const uint32_t a_lbo = (uint32_t)a_rows * 16, b_lbo = (uint32_t)NE * 16;
    const uint32_t a_plane32 = (uint32_t)L.a_plane, b_plane32 = (uint32_t)L.b_plane;
    const uint64_t a_desc0 = make_kmajor_desc(smem_u32(sA), a_lbo, 128);
    const uint64_t b_desc0 = make_kmajor_desc(smem_u32(sB), b_lbo, 128);
    MT_TC_TIMER();  // 0: wait bready, 1: issue
    for (int k = 0;; ++k) {  // k counts the chunks that carry edges (and the terminator)
      // lane 0 alone reads the hand-over word: by the time the other lanes get here the producer may already
      // have posted the next chunk (or the terminator) -- a per-lane read would split the warp
      int b = 0;
      if (lane == 0) {
        mbar_wait(&bar_bready, k & 1, 30);
        b = s_mma_b;
      }
      b = __shfl_sync(0xffffffffu, b, 0);
      MT_TACC(0);
      if (b < 0) break;
      if (lane == 0) {
        tc_fence_after();
        // significant products of (hi+mid+lo) x (hi+mid+lo), small ones first: planes (a, b) = (0,2) (2,0) (1,1) (0,1)
        // (1,0) (0,0), two bits each, packed (a local array would live in local memory: an L2 trip per MMA)
        constexpr uint32_t kPa = 0u | (2u << 2) | (1u << 4) | (0u << 6) | (1u << 8) | (0u << 10);
        constexpr uint32_t kPb = 2u | (0u << 2) | (1u << 4) | (1u << 6) | (0u << 8) | (0u << 10);
        for (int t = 0; t < MT; ++t) {
          const uint32_t d = tmem_base + (uint32_t)((b * MT + t) * NE);
          uint32_t accum = 0;
#pragma unroll
          for (int q = 0; q < 6; ++q) {
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              // descriptors differ only in the start-address field (units of 16 bytes, no carry: < 2^14)
              const uint32_t a_off = ((kPa >> (2 * q)) & 3u) * a_plane32 + (uint32_t)(2 * ks) * a_lbo + (uint32_t)t * 128 * 16;
              const uint32_t b_off = ((kPb >> (2 * q)) & 3u) * b_plane32 + (uint32_t)(2 * ks) * b_lbo;
              umma_bf16(d, a_desc0 + (uint64_t)(a_off >> 4), b_desc0 + (uint64_t)(b_off >> 4), idesc, accum);
              accum = 1;
            }
          }
        }
        umma_commit(&bar_full[b]);
        umma_commit(&bar_bfree);
      }
      __syncwarp();
      MT_TACC(1);
    }
    MT_TC_TIMER_FLUSH();
  } else if (warp == 2 || warp == 3) {
    // ================================================================ TMA gathers of the sender rows (a gather4 costs
    // its issuing warp ~250 cycles per active lane).  One-tile parts have 256-column chunks = 64 gathers: warps 2 and 3
    // take the even / odd groups of 4 columns (-5 %); with more tiles (<= 32 gathers per chunk) a second active
    // producer warp only takes issue slots from the consumers (+3-5 %), so warp 3 idles there.
    const int ngw = MT == 1 ? 2 : 1;
    const int gw = warp == 2 ? 0 : 1;
    if (gw < ngw) {
    const CUtensorMap* map = &maps.m[part_id];
    const uint32_t xrow_bytes = (uint32_t)P.x_cols * 4;
    MT_TC_TIMER();  // 0: wait go, 1: issue
    for (int k = 0;; ++k) {
      const int b = k & 1;
      const TcMeta& M = *reinterpret_cast<const TcMeta*>(sMeta + b * kMetaBytes);
      if (lane == 0) mbar_wait(&bar_go[b], (k >> 1) & 1, 50 + b);
      __syncwarp();
      MT_TACC(0);
      const int nn = M.nnodes, ncols = M.ncols, pc0 = M.pc0;
      if (nn < 0) break;
      unsigned char* xs = smem + L.x_off + (size_t)b * L.x_buf;
      for (int g = ngw * lane + gw; g < (ncols >> 2); g += 32 * ngw) {
        const int4 r = *reinterpret_cast<const int4*>(p.src_pad + pc0 + 4 * g);
        tma_gather4(xs + (size_t)(4 * g) * xrow_bytes, map, P.x_lo, r.x, r.y, r.z, r.w, &bar_full[b]);
      }
      MT_TACC(1);
    }
    MT_TC_TIMER_FLUSH();
    }
  } else {
    // ================================================================ consumers
    const int q = warp & 3;
    const int nbiq = P.q_count[q];
    MT_TC_TIMER();  // 0: wait full, 1: units, 7: units processed
    for (int k = 0;; ++k) {
      const int b = k & 1;
      // one lane waits (a warp-wide poll would flood the shared-memory pipe the producers' LDS need)
      if (lane == 0) mbar_wait(&bar_full[b], (k >> 1) & 1, 40 + b);
      __syncwarp();
      MT_TACC(0);
      tc_fence_after();
      const TcMeta& M = *reinterpret_cast<const TcMeta*>(sMeta + b * kMetaBytes);
      const int nn = M.nnodes;
      if (nn < 0) break;
      TcUnit u;
      u.tstage = tmem_base + (uint32_t)(b * MT * NE);
      u.quarter = q;
      u.ne = NE;
      u.xs = reinterpret_cast<const float*>(smem + L.x_off + (size_t)b * L.x_buf);
      u.xstride = P.x_cols;
      u.ys = reinterpret_cast<const float*>(smem + L.y_off + (size_t)b * L.y_buf);
      u.ystride = ystride;
      const int num_units = nbiq * nn;
      while (true) {
        int unit = 0;
        if (lane == 0) unit = atomicAdd(&s_cnt[b][q], 1);
        unit = __shfl_sync(0xffffffffu, unit, 0);
        if (unit >= num_units) break;
        const int si = unit / nn, nj = unit - si * nn;
        const int bi = sQ[q * kTcMaxBI + si];
        const int4 h0 = *reinterpret_cast<const int4*>(sHdr + bi * 8);
        const int4 h1 = *reinterpret_cast<const int4*>(sHdr + bi * 8 + 4);
        u.mask = (unsigned)h0.w;
        u.nch = h0.z;
        u.slot[0] = h1.y; u.slot[1] = h1.z; u.slot[2] = h1.w;
        u.lt = sLane[bi * 32 + lane];
        u.cb = M.cb[nj];
        u.ngrp = M.ngrp[nj];
        u.out = p.out + (size_t)M.node_id[nj] * p.out_dim;
        u.inv_den = M.inv_den[nj];
        u.first = M.first[nj] != 0;
        __syncwarp();
        switch (h0.x) {
#define MT_TC_CASE(ID) \
  case ID:             \
    tc_unit_dispatch<ID>(u, h0.y, lane); \
    break;
          MT_FOR_EACH_BUNDLE_L2(MT_TC_CASE)
          default:
            if constexpr (LMAXK > 2) {
              switch (h0.x) {
                MT_FOR_EACH_BUNDLE_GT2(MT_TC_CASE)
                default: break;
              }
            }
            break;
#undef MT_TC_CASE
        }
        __syncwarp();
        if (_tm) _ta[7] += 16;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_empty[b]);
      MT_TACC(1);
    }
    MT_TC_TIMER_FLUSH();
  }
  // ---------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace mt
