// LightpathGNN eval forward with EVERY node of a graph as the LUT (lightpath under test), one pass over the graph.
//
// Semantics: for a batch with N nodes, row i of out [N,3] is what the reference LightpathGNN.forward under eval()
// returns for node i's graph, given a copy of that graph in which node i's flag column x[:, is_lut_index] is 1.0
// and every other node's flag column is 0.0.  Whatever the stored flag column holds has no effect.  Rows are in
// node order; the graph of row i is batch[i].
//
// Why one pass suffices: the model has one GAT layer and, in eval mode, BatchNorm is a per-node affine, so the
// prediction for node v as LUT depends only on x_v with its flag set to 1 (its attention query d_v and its appended
// self loop) and on x_j with the flag set to 0 for every in-neighbour j.
//
//   work item = a TILE of 12 consecutive graphs of one batch, walked over the same descriptor array as
//   qot_lightpath_infer_stream; one CTA per SM loops over tiles bid, bid + grid, ...; warp w of the CTA takes graph
//   w of each of its tiles, with no block-level synchronisation after the prologue.
//
//   fast path (n <= kEnMaxN, E_g <= kEnMaxE, every message source inside the graph): the warp stages the graph's x
//     (flag column zeroed) and the destination row of its edges in shared memory, builds the graph's
//     destination-sorted in-CSR there (self loops dropped, one extra slot per row for the appended self loop):
//       unverified layout: a stable counting sort of the edges by destination -- a row's messages in edge order;
//       QOT_LP_SYMMETRIC_BY_SOURCE: the in-neighbours of v are the destinations of v's own out-run
//         [#{dst < v}, #{dst <= v}), ranked ascending -- the source row is never read.
//     On a verified layout both give every row its sources in ascending order: bit-identical results.
//     Then 4-head attention per node (attn_consume over the row, node v's own flag and d_v taken with flag = 1).
//   generic path (larger graphs, sources outside the graph): lut_row_global with the XAsLut accessor, row by row
//     straight from global memory, inside the same launch.
//   head: each z row (20 floats) is staged in the warp's 16-row buffer; a full buffer (rows may come from several
//     graphs) goes through head_rows16_tf32x3 -- the readout head of lp_stream_head_kernel on mma.sync, 3xTF32.
//
// Deterministic: no float atomics, fixed reduction order, the path a graph takes depends only on its sizes and
// edge endpoints (not on the flag column, not on the layout flag).  Every index read from the batch is bounds
// checked; malformed graph offsets set status bit 0 and the graph's rows are not written.
#include <algorithm>

#include "lightpath_common.cuh"

namespace qot {

constexpr int kEnTG = 12;                  // graphs per tile
constexpr int kEnWarps = 12;               // warp w takes graph w of a tile (12 warps: 168 registers, no spills)
constexpr int kEnThreads = 32 * kEnWarps;
constexpr int kEnMaxN = 128;               // fast path: nodes of a graph staged per warp
constexpr int kEnMaxE = 512;               // fast path: edges of a graph staged per warp
constexpr int kEnZPitch = kHeads * kF;     // 20 floats per staged z row: rows g8 / g8 + 8 of the head hit 32 banks
static_assert(kEnTG == kEnWarps, "one graph of each tile per warp");

struct EnWarpSmem {
  float x[kEnMaxN * kF];                   // graph's x, flag column zeroed
  int rs[kEnMaxN + 1];                     // in-CSR row starts (row v: rs[v] .. rs[v] + rl[v], then the self loop)
  int rl[kEnMaxN];                         // messages of row v without the self loop
  int msg[kEnMaxE + kEnMaxN];              // graph-local sources
  short ed[kEnMaxE];                       // graph-local destination of every edge (-1: outside the graph)
  float z[16 * kEnZPitch];                 // staged z rows of the head
  long long orow[16];                      // where each staged row's 3 outputs go
  float gz[32];                            // generic path: z of one row (slot h*8+f)
};
struct EnSmem {
  float4 frag[kStHeadFrag4];               // B1f | B2f fragment tables of the mma.sync head
  EnWarpSmem w[kEnWarps];
};
static_assert(sizeof(EnSmem) + 16 <= 227 * 1024, "lp_every_node_kernel: shared memory over the 227 KB block limit");

// Every access to the block's shared memory goes through this accessor, so the compiler sees the shared window and
// emits LDS / STS instead of generic loads and stores.
extern __shared__ __align__(16) char en_smem_raw[];
__device__ __forceinline__ EnSmem& en_smem() { return *reinterpret_cast<EnSmem*>(en_smem_raw); }

// z rows staged in the warp's buffer -> out rows (cnt <= 16).  Not inlined: the head's accumulators then do not
// share a register allocation with the attention loop.
__device__ __noinline__ void en_flush(int w, int cnt, const float* __restrict__ prep, int lane) {
  EnSmem& sm = en_smem();
  EnWarpSmem& ws = sm.w[w];
  const int g8 = lane >> 2, t4 = lane & 3;
  const bool va = g8 < cnt, vb = g8 + 8 < cnt;
  float oa, ob;
  head_rows16_tf32x3(sm.frag, sm.frag + 16 * 32, ws.z + g8 * kEnZPitch, ws.z + (g8 + 8) * kEnZPitch, va, vb, prep,
                     lane, oa, ob);
  if (t4 < QOT_OUT) {
    if (va) reinterpret_cast<float*>(ws.orow[g8])[t4] = oa;
    if (vb) reinterpret_cast<float*>(ws.orow[g8 + 8])[t4] = ob;
  }
  __syncwarp();
}

// Builds the in-CSR of a staged graph (n nodes, ne edges, destinations in ws.ed).  Returns false when a message
// source lies outside the graph (the graph then takes the generic path).
template <bool kSym>
__device__ __forceinline__ bool en_build_csr(EnWarpSmem& ws, const int64_t* __restrict__ esrc, int64_t n0, int64_t N,
                                             int n, int ne, int lane) {
  for (int v = lane; v <= n; v += 32) ws.rs[v] = 0;
  __syncwarp();
  // in-degree histogram, integer shared atomics (exact).  kSym: every in-graph destination (the out-run lengths);
  // otherwise the message count: destination in the graph, source != destination, source inside [0, N).
  bool outside = false;
  for (int e = lane; e < ne; e += 32) {
    const int d = ws.ed[e];
    if (d < 0) continue;
    if constexpr (kSym) {
      atomicAdd(&ws.rs[d + 1], 1);
    } else {
      const int64_t s = esrc[e];
      if (s == n0 + d || static_cast<uint64_t>(s) >= static_cast<uint64_t>(N)) continue;
      if (s < n0 || s >= n0 + n) outside = true;
      atomicAdd(&ws.rs[d + 1], 1);
    }
  }
  if (__any_sync(kFull, outside)) return false;
  __syncwarp();
  // exclusive prefix of the counts: run / row starts
  int carry = 0;
  for (int b0 = 0; b0 <= n; b0 += 32) {
    const int v = b0 + lane;
    int c = v <= n ? ws.rs[v] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int up = __shfl_up_sync(kFull, c, o);
      if (lane >= o) c += up;
    }
    if (v <= n) ws.rs[v] = c + carry;
    carry += __shfl_sync(kFull, c, 31);
  }
  __syncwarp();
  if constexpr (kSym) {
    // row v = the out-run of v, self loops dropped, ranked ascending (a verified layout has no duplicate pairs).
    // rs[v] is the run start; the row is written at rs[v] + v (one extra slot per row for the self loop).
    for (int v = lane; v < n; v += 32) {
      const int r0 = ws.rs[v], r1 = ws.rs[v + 1];
      int kept = 0;
      for (int e = r0; e < r1; ++e) {
        const int d = ws.ed[e];
        if (d == v) continue;
        int rank = 0;
        for (int f = r0; f < r1; ++f) {
          const int df = ws.ed[f];
          rank += (df != v) & (df < d);
        }
        ws.msg[r0 + v + rank] = d;
        ++kept;
      }
      ws.rl[v] = kept;
      ws.msg[r0 + v + kept] = v;                 // the appended self loop comes last
    }
    __syncwarp();
    for (int v = lane; v <= n; v += 32) ws.rs[v] += v;   // rows start at run start + v
    return true;
  } else {
    // stable placement in edge order: 32 edges per step, lanes with the same destination ranked by lane
    for (int v = lane; v < n; v += 32) {
      ws.rl[v] = ws.rs[v + 1] - ws.rs[v];
      ws.rs[v] += v;                              // one extra slot per row
    }
    if (lane == 0) ws.rs[n] += n;
    __syncwarp();
    for (int v = lane; v < n; v += 32) ws.msg[ws.rs[v] + ws.rl[v]] = v;   // the self loop, last in the row
    // rl doubles as the placement cursor: it ends at the row's message count again
    int* cur = ws.rl;
    for (int v = lane; v < n; v += 32) cur[v] = 0;
    __syncwarp();
    for (int eb = 0; eb < ne; eb += 32) {
      const int e = eb + lane;
      int d = -1;
      int s = 0;
      if (e < ne) {
        d = ws.ed[e];
        if (d >= 0) {
          const int64_t sg = esrc[e];
          if (sg == n0 + d || static_cast<uint64_t>(sg) >= static_cast<uint64_t>(N)) d = -1;
          else s = static_cast<int>(sg - n0);
        }
      }
      const unsigned peers = __match_any_sync(kFull, d);
      if (d >= 0) {
        const int rank = __popc(peers & ((1u << lane) - 1u));
        ws.msg[ws.rs[d] + cur[d] + rank] = s;
      }
      __syncwarp();
      if (d >= 0 && lane == 31 - __clz(peers)) cur[d] += __popc(peers);
      __syncwarp();
    }
    return true;
  }
}

// graph g of batch d: every node's z row into the warp's head buffer (zc rows staged); returns the new zc
template <bool kSym>
__device__ __forceinline__ int en_graph(const qot_lp_batch_t& d, int64_t g, const float* __restrict__ prep, int lut_col,
                                        int w, int zc, int lane) {
  EnSmem& sm = en_smem();
  EnWarpSmem& ws = sm.w[w];
  const int64_t N = d.N, E = d.E;
  const int64_t n0 = d.ptr[g], n1 = d.ptr[g + 1], e0 = d.edge_ptr[g], e1 = d.edge_ptr[g + 1];
  if (!(n0 >= 0 && n1 >= n0 && n1 <= N && e0 >= 0 && e1 >= e0 && e1 <= E)) {
    if (lane == 0) atomicOr(d.status, 1);
    return zc;
  }
  const int64_t* __restrict__ esrc = d.edge_index;
  const int64_t* __restrict__ edst = d.edge_index + E;
  const int n = static_cast<int>(n1 - n0);
  const int64_t ne64 = e1 - e0;
  bool fast = n <= kEnMaxN && ne64 <= kEnMaxE;
  if (fast) {
    const int ne = static_cast<int>(ne64);
    for (int i = lane; i < n * kF; i += 32) ws.x[i] = (i % kF == lut_col) ? 0.f : d.x[n0 * kF + i];
    bool out_of_graph = false;
    for (int e = lane; e < ne; e += 32) {
      const int64_t dd = edst[e0 + e];
      const bool in = dd >= n0 && dd < n1;
      ws.ed[e] = in ? static_cast<short>(dd - n0) : static_cast<short>(-1);
      out_of_graph |= !in;
    }
    __syncwarp();
    // kSym: a destination outside the graph breaks the run structure (the layout was not what was verified)
    if (kSym && __any_sync(kFull, out_of_graph)) fast = false;
    if (fast) fast = en_build_csr<kSym>(ws, esrc + e0, n0, N, n, ne, lane);
    __syncwarp();
  }
  const int h = lane & 3;
  float As[kF], Ad[kF];
#pragma unroll
  for (int k = 0; k < kF; ++k) {
    As[k] = __ldg(prep + kOffAsrc + k * kHeads + h);
    Ad[k] = __ldg(prep + kOffAdst + k * kHeads + h);
  }
  for (int v = 0; v < n; ++v) {
    float* zr = ws.z + zc * kEnZPitch;
    if (fast) {
      const float* sx = ws.x;
      auto xf = [&](int j, int k) { return (k == lut_col && j == v) ? 1.0f : sx[j * kF + k]; };
      float d_v = 0.f;
#pragma unroll
      for (int k = 0; k < kF; ++k) d_v = fmaf(xf(v, k), Ad[k], d_v);
      AttnState st;
      attn_consume(st, ws.msg + ws.rs[v], ws.rl[v] + 1, xf, As, d_v, lane);
      attn_finish<kF>(st, zr, lane);                      // [h][f]: the head's row layout
    } else {
      lut_row_global<false>(XAsLut{d.x, n0 + v, lut_col}, esrc, edst, e0, e1, N, n0 + v, prep, nullptr,
                            reinterpret_cast<int*>(ws.msg), ws.gz, nullptr, lane);
      if (lane < kHeads * kF) zr[lane] = ws.gz[(lane / kF) * 8 + lane % kF];
    }
    if (lane == 0) ws.orow[zc] = reinterpret_cast<long long>(d.out + (n0 + v) * QOT_OUT);
    __syncwarp();
    if (++zc == 16) {
      en_flush(w, 16, prep, lane);
      zc = 0;
    }
  }
  return zc;
}

template <bool kSym>
__global__ void __launch_bounds__(kEnThreads, 1)
lp_every_node_kernel(const qot_lp_batch_t* __restrict__ batches, int n_batches, int64_t tiles_per_batch,
                     int64_t total_tiles, const float* __restrict__ prep, int lut_col) {
  EnSmem& sm = en_smem();
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  for (int i = tid; i < kStHeadFrag4; i += kEnThreads) sm.frag[i] = __ldg(reinterpret_cast<const float4*>(prep + kOffB1f) + i);
  __syncthreads();
  const int64_t base = batches[0].tile0;
  int zc = 0;                                   // rows staged in this warp's head buffer
  for (int64_t T = blockIdx.x; T < total_tiles; T += gridDim.x) {
    const int b = st_batch_of(batches, n_batches, tiles_per_batch, base, base + T);
    const qot_lp_batch_t& d = batches[b];
    const int64_t g = (base + T - d.tile0) * kEnTG + w;
    if (g < 0 || g >= d.B) continue;
    zc = en_graph<kSym>(d, g, prep, lut_col, w, zc, lane);
  }
  if (zc) en_flush(w, zc, prep, lane);
}

}  // namespace qot

using namespace qot;

extern "C" int64_t qot_lightpath_every_node_tiles(int64_t B) { return B > 0 ? cdiv(B, kEnTG) : 0; }

// `batches`: DEVICE array of n_batches descriptors with tile0 filled (tile0[b+1] = tile0[b] +
// qot_lightpath_every_node_tiles(B_b); tile0[0] is arbitrary, so a sub-range of a longer array can be launched).
// Reads x, edge_index, ptr, edge_ptr, N, E, B, out (>= N rows), status, tile0 of every descriptor.
extern "C" int qot_lightpath_infer_every_node(const qot_lp_batch_t* batches, int32_t n_batches, int64_t total_tiles,
                                              int64_t uniform_tiles, const float* prepared, int32_t is_lut_index,
                                              int32_t flags, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  QOT_REQUIRE(batches && n_batches > 0 && total_tiles >= 0 && uniform_tiles >= 0,
              "qot_lightpath_infer_every_node: bad argument");
  QOT_REQUIRE(prepared && (reinterpret_cast<uintptr_t>(prepared) & 15) == 0,
              "qot_lightpath_infer_every_node: prepared must be 16-byte aligned");
  QOT_REQUIRE(is_lut_index >= 0 && is_lut_index < kF, "qot_lightpath_infer_every_node: is_lut_index out of range");
  QOT_REQUIRE((flags & ~QOT_LP_SYMMETRIC_BY_SOURCE) == 0, "qot_lightpath_infer_every_node: unknown flag");
  if (total_tiles == 0) return QOT_OK;
  const bool sym = (flags & QOT_LP_SYMMETRIC_BY_SOURCE) != 0;
  static std::atomic<unsigned long long> done{0};
  constexpr int smem = static_cast<int>(sizeof(EnSmem));
  if (int rc = once_per_device(done, [] {
        QOT_CUDA(cudaFuncSetAttribute(lp_every_node_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        QOT_CUDA(cudaFuncSetAttribute(lp_every_node_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        return static_cast<int>(QOT_OK);
      }))
    return rc;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, total_tiles));
  if (sym)
    lp_every_node_kernel<true><<<grid, kEnThreads, smem, stream>>>(batches, n_batches, uniform_tiles, total_tiles,
                                                                   prepared, is_lut_index);
  else
    lp_every_node_kernel<false><<<grid, kEnThreads, smem, stream>>>(batches, n_batches, uniform_tiles, total_tiles,
                                                                    prepared, is_lut_index);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}
