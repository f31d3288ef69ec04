// LightpathGNN network-state queries: candidate lightpaths, reconfigurations, change sets, placements and sequential
// provisioning evaluated against a resident network state without rebuilding the state's graph.
//
// Why no rebuild is needed: the model has one GAT layer and eval-mode BatchNorm is a per-node affine, so a row depends
// only on its node and its in-neighbours.  Placing a lightpath adds exactly the edges new <-> j for the lightpaths j
// that share a link with it at 0 < |df| < freq_threshold, and removing one drops its edges; every other row of the
// graph is unchanged.
//
//   lp_channel_map_kernel (once per state): chan_node [S, L, Q] = state-batch node index of the lightpath on each
//     channel, -1 on a free channel (occupancy and conn_id truncation as in to_graph.cu).
//
// The query kernels are persistent, one warp per query, and built from the same pieces, each defined once below:
//   cd_bad_route, cd_sample_nodes  a route (its link_ptr range, every link in [0, L)) and a sample's node range;
//   cd_df_hit                      to_graph.cu's fp64 edge test: some slot of [c0, c0 + cw) at 0 < |df| < threshold;
//   cd_scan                        the chan_node rows of a route, cd_df_hit against every channel of a known lightpath,
//                                  neighbours into a 256-bit per-warp mask (a state sample holds at most
//                                  QOT_TG_MAX_NODES lightpaths); the lightpaths a query removes count as free;
//   cd_old_nbrs                    a removed lightpath's old neighbours: the destinations of its out-run;
//   cd_rank                        a mask's bits in ascending order (the order of rows and messages);
//   cd_xrow                        a new lightpath's scaled x row [freq, is_lut = 1, mod_order, num_spans, path_len];
//   cd_in_row                      j's in-row of the state graph: the destinations of j's out-run in the source-sorted
//                                  edge list, j's self loop and the removed lightpaths dropped;
//   cd_head_prologue, cd_row       the head: every z row is staged in the warp's 16-row buffer and goes through
//                                  head_rows16_tf32x3 (the mma.sync head of every-node mode) in cd_flush;
//   cd_clear_impact                the empty result past the emitted impact rows: node -1, kind 0, NaN QoT.
// A new lightpath's row is: query flag 1, its new neighbours ascending (flag 0), its appended self loop.  The impact
// row of neighbour j is: query flag 1, j's in-row (flag 0), the new lightpath (flag 0) if j is a new neighbour, j's
// self loop.  Because every kernel builds its rows from these pieces in this message order, an insertion through
// qot_lightpath_reconfigure is bit-identical to a candidate, a set of one change to a reconfiguration, and a
// placement's rows to the candidate on the same slots.
//
// Deterministic: integer mask bits only, fixed message order, no float atomics.  A malformed query gets status bits
// and NaN rows; it never faults and never stops the launch.
#include <algorithm>
#include <climits>
#include <type_traits>

#include "lightpath_common.cuh"

namespace qot {

// ------------------------------------------------------------------------------------------------ channel map
constexpr int kCmThreads = 256;

__global__ void __launch_bounds__(kCmThreads)
lp_channel_map_kernel(const float* __restrict__ data, qot_lp_graph_cfg_t cfg, const int64_t* __restrict__ node_ptr,
                      const int64_t* __restrict__ conn_ids, int64_t N, int32_t* __restrict__ chan_node,
                      int32_t* __restrict__ status) {
  __shared__ int64_t sconn[QOT_TG_MAX_NODES];
  const int tid = threadIdx.x;
  const int64_t s = blockIdx.x;
  const int LQ = cfg.L * cfg.Q;
  const float* __restrict__ d = data + s * static_cast<int64_t>(cfg.F) * LQ;
  int32_t* __restrict__ row = chan_node + s * LQ;
  const int64_t n0 = node_ptr[s], n1 = node_ptr[s + 1];
  const bool ok = n0 >= 0 && n1 >= n0 && n1 <= N && n1 - n0 <= QOT_TG_MAX_NODES;
  const int n = ok ? static_cast<int>(n1 - n0) : 0;
  for (int r = tid; r < n; r += kCmThreads) sconn[r] = conn_ids[n0 + r];
  __syncthreads();
  bool missing = !ok;
  for (int ch = tid; ch < LQ; ch += kCmThreads) {
    bool occ = false;
    for (int f = 0; f < cfg.F; ++f) occ |= d[static_cast<int64_t>(f) * LQ + ch] != 0.f;
    int32_t v = -1;
    if (occ) {
      const int64_t c = static_cast<int>(d[static_cast<int64_t>(cfg.i_conn) * LQ + ch]);   // int(): toward zero
      v = INT_MIN;                                       // occupied by a lightpath the node list does not know
      for (int r = 0; r < n; ++r)
        if (sconn[r] == c) { v = static_cast<int32_t>(n0 + r); break; }
      missing |= v == INT_MIN;
    }
    row[ch] = v;
  }
  if (missing && status) atomicOr(status, 1);
}

// ------------------------------------------------------------------------------------------------ candidates
constexpr int kCdWarps = 12;                 // 12 warps: the register budget of every-node mode, no spills
constexpr int kCdThreads = 32 * kCdWarps;
constexpr int kCdMaxN = QOT_TG_MAX_NODES;          // lightpaths of a state sample: bits of the neighbour mask
constexpr int kCdMaskWords = kCdMaxN / 32;
constexpr int kCdMsgCap = kCdMaxN + 8;             // in-row of a neighbour (<= kCdMaxN) + candidate + self loop
constexpr int kCdZPitch = kHeads * kF;             // 20 floats per staged z row (as in every-node mode)
constexpr int kCand = -1;                          // message index of the candidate itself
static_assert(kCdMaskWords <= 32, "one mask word per lane");

struct CdWarpSmem {
  float z[16 * kCdZPitch];                 // staged z rows of the head
  long long orow[16];                      // where each staged row's 3 outputs go
  int nbr[kCdMaxN + 1];                    // impact rows (sample-local, ascending), then the candidate's self loop
  int msg[kCdMsgCap];                      // message list of one row
  unsigned mask[kCdMaskWords];             // neighbour bits of the new placement
  unsigned omask[kCdMaskWords];            // old neighbour bits of the moved lightpath (reconfiguration only)
  float cx[8];                             // the candidate's scaled x row
};
struct CdSmem {
  float4 frag[kStHeadFrag4];               // B1f | B2f fragment tables of the mma.sync head
  CdWarpSmem w[kCdWarps];
};
static_assert(sizeof(CdSmem) + 16 <= 227 * 1024, "lp_candidate_kernel: shared memory over the 227 KB block limit");

extern __shared__ __align__(16) char cd_smem_raw[];
__device__ __forceinline__ CdSmem& cd_smem() { return *reinterpret_cast<CdSmem*>(cd_smem_raw); }

// x of a message source: sample-local node j of the state (x read from global memory) or the candidate (kCand);
// the flag column is 1.0 for `lut` and 0.0 for every other node.
struct CdX {
  const float* __restrict__ xs;            // state x of the sample's first node
  const float* cx;
  int lut, col;
  __device__ __forceinline__ float operator()(int j, int k) const {
    if (k == col) return j == lut ? 1.0f : 0.0f;
    return j == kCand ? cx[k] : __ldg(xs + static_cast<int64_t>(j) * kF + k);
  }
};

struct CdArgs {
  qot_lp_graph_cfg_t cfg;
  int64_t S, N, E, K, n_links;
  const double* freqs;
  const float* x;
  const int64_t* node_ptr;
  const int64_t* rowptr;
  const int64_t* edst;                     // destination row of the state's source-sorted edge_index
  const int32_t* chan_node;
  const int64_t* node;                     // moved lightpath of each change (kMove only)
  const int64_t* sample;
  const int64_t* link_ptr;
  const int32_t* links;
  const int32_t* q0;
  const int32_t* width;
  const float* feat;
  const float* prep;
  int lut_col, max_impact;
  float* out;
  int32_t* status;
  int32_t* n_impact;
  int64_t* impact_node;
  int8_t* impact_kind;                     // optional (kMove only)
  float* impact_out;
};

// The helpers below read L, Q, the threshold and max_impact from the kernel parameters where they use them: hoisted
// into registers, those values spill in the change-set kernel.

// the head's fragment tables into shared memory (published by the caller's next block barrier) and this lane's head
// column of the attention vectors into registers
__device__ __forceinline__ void cd_head_prologue(const float* __restrict__ prep, float (&As)[kF], float (&Ad)[kF],
                                                 int tid) {
  CdSmem& sm = cd_smem();
  for (int i = tid; i < kStHeadFrag4; i += kCdThreads)
    sm.frag[i] = __ldg(reinterpret_cast<const float4*>(prep + kOffB1f) + i);
  const int h = tid & 3;
#pragma unroll
  for (int k = 0; k < kF; ++k) {
    As[k] = __ldg(prep + kOffAsrc + k * kHeads + h);
    Ad[k] = __ldg(prep + kOffAdst + k * kHeads + h);
  }
}

__device__ __noinline__ void cd_flush(int w, int cnt, const float* __restrict__ prep, int lane) {
  CdSmem& sm = cd_smem();
  CdWarpSmem& ws = sm.w[w];
  const int g8 = lane >> 2, t4 = lane & 3;
  const bool va = g8 < cnt, vb = g8 + 8 < cnt;
  float oa, ob;
  head_rows16_tf32x3(sm.frag, sm.frag + 16 * 32, ws.z + g8 * kCdZPitch, ws.z + (g8 + 8) * kCdZPitch, va, vb, prep,
                     lane, oa, ob);
  if (t4 < QOT_OUT) {
    if (va) reinterpret_cast<float*>(ws.orow[g8])[t4] = oa;
    if (vb) reinterpret_cast<float*>(ws.orow[g8 + 8])[t4] = ob;
  }
  __syncwarp();
}

// attention of query node q over msg[0, M) into staged z row zc, whose outputs go to `dst`; a full buffer of 16 rows
// goes to `flush(16)`.  Returns the rows staged.
template <typename XF, typename Flush>
__device__ __forceinline__ int cd_row(CdWarpSmem& ws, int zc, const int* msg, int M, int q, const XF& xf,
                                      const float (&As)[kF], const float (&Ad)[kF], float* dst, const Flush& flush,
                                      int lane) {
  float d_q = 0.f;
#pragma unroll
  for (int k = 0; k < kF; ++k) d_q = fmaf(xf(q, k), Ad[k], d_q);
  AttnState st;
  attn_consume(st, msg, M, xf, As, d_q, lane);
  attn_finish<kF>(st, ws.z + zc * kCdZPitch, lane);
  if (lane == 0) ws.orow[zc] = reinterpret_cast<long long>(dst);
  __syncwarp();
  if (++zc == 16) {
    flush(16);
    zc = 0;
  }
  return zc;
}

// ranks the set bits of a 256-bit mask (lane t < 8 holds word t) ascending into dst[0, count); returns the count
__device__ __forceinline__ int cd_rank(unsigned mw, int* dst, int lane) {
  int pos = __popc(mw);
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int up = __shfl_up_sync(kFull, pos, o);
    if (lane >= o) pos += up;
  }
  const int cnt = __shfl_sync(kFull, pos, 31);
  pos -= __popc(mw);
  for (unsigned m = mw; m; m &= m - 1) dst[pos++] = 32 * lane + __ffs(m) - 1;
  return cnt;
}

// to_graph.cu's edge test, in fp64: some slot c of [c0, c0 + cw) at 0 < |freqs[c] - fq| < thr
__device__ __forceinline__ bool cd_df_hit(const double* freqs, double fq, int c0, int cw, double thr) {
  bool hit = false;
  for (int c = c0; c < c0 + cw && !hit; ++c) {
    const double df = fabs(freqs[c] - fq);
    hit = df < thr && df > 0.0;
  }
  return hit;
}

// removes no lightpath: the predicate of cd_scan and cd_in_row for candidates and placements
struct CdNone {
  __device__ __forceinline__ bool operator()(int) const { return false; }
};

// the new neighbours of placement [c0, c0 + cw) on route links[p0, p1) of sample s (nodes [n0, n0 + n)): the known
// lightpath on every other channel of the route's chan_node rows that passes cd_df_hit sets its bit in `mask`.  A
// channel of a lightpath `removed(j)` names (sample-local) counts as free.  Returns this lane's status bits:
// QOT_CAND_OCCUPIED (a channel of the placement is taken), QOT_CAND_BAD_STATE (an owner outside the sample).
template <typename Removed>
__device__ __forceinline__ int cd_scan(const CdArgs& a, int64_t s, int64_t n0, int n, int64_t p0, int64_t p1, int c0,
                                       int cw, unsigned* mask, const Removed& removed, int lane) {
  bool occ = false, bad = false;
  for (int64_t e = p0; e < p1; ++e) {
    const int32_t* __restrict__ row = a.chan_node + (s * a.cfg.L + a.links[e]) * a.cfg.Q;
    for (int q = lane; q < a.cfg.Q; q += 32) {
      const int32_t v = row[q];
      if (v == -1) continue;                                    // free
      const int64_t j = v - n0;
      const bool inside = v >= 0 && j >= 0 && j < n;
      if (inside && removed(static_cast<int>(j))) continue;
      if (q >= c0 && q < c0 + cw) { occ = true; continue; }
      if (v < -1) continue;                                     // occupied by an unknown lightpath: no edge
      if (!inside) { bad = true; continue; }
      if (cd_df_hit(a.freqs, a.freqs[q], c0, cw, a.cfg.freq_threshold)) atomicOr(&mask[j >> 5], 1u << (j & 31));
    }
  }
  return (occ ? QOT_CAND_OCCUPIED : 0) | (bad ? QOT_CAND_BAD_STATE : 0);
}

// the old neighbours of sample-local node jm: the destinations of its out-run, self loop dropped, into `mask`; false
// (on this lane) when the run is malformed or leaves the sample
__device__ __forceinline__ bool cd_old_nbrs(const CdArgs& a, int64_t n0, int n, int jm, unsigned* mask, int lane) {
  const int64_t r0 = a.rowptr[n0 + jm], r1 = a.rowptr[n0 + jm + 1];
  if (!(r0 >= 0 && r1 >= r0 && r1 <= a.E)) return false;
  bool ok = true;
  for (int64_t e = r0 + lane; e < r1; e += 32) {
    const int64_t dg = a.edst[e] - n0;
    if (dg < 0 || dg >= n) ok = false;
    else if (dg != jm) atomicOr(&mask[dg >> 5], 1u << (dg & 31));
  }
  return ok;
}

// sample-local node j's in-row of the state graph: the destinations of j's out-run in the source-sorted edge list, in
// edge order, without j's self loop and the nodes `drop` names, into msg.  Returns their count, or -1 (warp-uniform)
// when the run is malformed, longer than a sample or leaves the sample.  kGather = false: the check alone.
template <bool kGather = true, typename Drop = CdNone>
__device__ __forceinline__ int cd_in_row(const CdArgs& a, int64_t n0, int n, int j, int* msg, int lane,
                                         const Drop& drop = Drop()) {
  const int64_t r0 = a.rowptr[n0 + j], r1 = a.rowptr[n0 + j + 1];
  bool bad = !(r0 >= 0 && r1 >= r0 && r1 <= a.E && r1 - r0 <= kCdMaxN);
  int m = 0;
  if (!bad)
    for (int64_t eb = r0; eb < r1; eb += 32) {
      const int64_t e = eb + lane;
      const int64_t dg = e < r1 ? a.edst[e] - n0 : -1;
      const bool inside = dg >= 0 && dg < n;
      bad |= e < r1 && !inside;
      if (kGather) {
        const bool keep = inside && dg != j && !drop(static_cast<int>(dg));
        const unsigned ball = __ballot_sync(kFull, keep);
        if (keep) msg[m + __popc(ball & ((1u << lane) - 1u))] = static_cast<int>(dg);
        m += __popc(ball);
      }
    }
  return __any_sync(kFull, bad) ? -1 : m;
}

// a new lightpath's x row [freq, is_lut, mod_order, num_spans, path_len] into cx: on lane t < 4, raw() gives raw
// feature t (freq, mod_order, num_spans, path_len) as float32, scaled min-max in fp64 and rounded to fp32 (dataset.py's
// scaling; feat_lo / feat_hi in that order); is_lut is 1, to_graph's value for a lightpath with unknown metrics
template <typename Raw>
__device__ __forceinline__ void cd_xrow(const CdArgs& a, float* cx, const Raw& raw, int lane) {
  if (lane < 4) {
    const double v = static_cast<double>(raw());
    cx[lane == 0 ? 0 : lane + 1] =
        static_cast<float>((v - a.cfg.feat_lo[lane]) / (a.cfg.feat_hi[lane] - a.cfg.feat_lo[lane]));
  }
  if (lane == 4) cx[1] = 1.0f;
}

// sample s's nodes [n0, n0 + n) of the state batch; false when node_ptr is malformed there or the sample holds more
// than kCdMaxN lightpaths (n0 is read either way)
__device__ __forceinline__ bool cd_sample_nodes(const CdArgs& a, int64_t s, int64_t& n0, int& n) {
  n0 = a.node_ptr[s];
  const int64_t n1 = a.node_ptr[s + 1];
  if (!(n0 >= 0 && n1 >= n0 && n1 <= a.N && n1 - n0 <= kCdMaxN)) return false;
  n = static_cast<int>(n1 - n0);
  return true;
}

// the route check, warp-uniform: links[p0, p1) is a non-empty range of `links` (an empty one for a teardown) whose
// links all lie in [0, L), and the caller's own checks `bad` (skipped for a teardown) pass; true when it fails.  L is
// cfg.L, passed in: the placement kernel keeps it in a register, and reading it here again spills there.
__device__ __forceinline__ bool cd_bad_route(const CdArgs& a, int L, int64_t p0, int64_t p1, bool tear, bool bad,
                                             int lane) {
  bad = tear ? !(p0 >= 0 && p0 <= a.n_links) : bad || !(p0 >= 0 && p1 > p0 && p1 <= a.n_links);
  if (!bad)
    for (int64_t e = p0 + lane; e < p1; e += 32) {
      const int l = a.links[e];
      bad |= l < 0 || l >= L;
    }
  return __any_sync(kFull, bad);
}

// the empty result in impact rows [from, MI) of output row k (MI = max_impact): node -1, kind 0 (when `kind`, the
// kernel's optional impact_kind), NaN QoT; written by threads t, t + stride, ...
__device__ __forceinline__ void cd_clear_impact(const CdArgs& a, int64_t k, int from, int MI, int8_t* kind, int t,
                                                int stride) {
  for (int i = from + t; i < MI; i += stride) {
    a.impact_node[k * MI + i] = -1;
    if (kind) kind[k * MI + i] = 0;
  }
  for (int i = from * QOT_OUT + t; i < MI * QOT_OUT; i += stride)
    a.impact_out[k * MI * QOT_OUT + i] = __int_as_float(0x7fc00000);
}

// lp_candidate_kernel, one warp per candidate: candidate k names a sample s_k of the state, a path, a slot range
// [q0_k, q0_k + width_k) used on every link of the path and its raw features (freq, mod_order, num_spans, path_len).
// sample' is s_k with the candidate written into those channels (a new conn_id, osnr = snr = ber = -1); out[k] is the
// candidate's row in sample''s lightpath graph with the flag column one-hot at the candidate, impact row i that of
// its i-th neighbour, neighbours ascending by state-batch node index.
//
// kMove = true (qot_lightpath_reconfigure): a change is a candidate that also names the lightpath j it moves (-1: a
// plain insertion, bit-identical to a candidate).  j's old channels count as free, its old neighbours go into a second
// 256-bit mask, and the impact rows are the union of both masks, ranked ascending, with kind bits old | new << 1.  j's
// row has its new neighbours (none for a teardown: NaN); impact row i drops j from i's in-row and takes j, with its
// new x, only if i is a new neighbour.
constexpr int kCdFatal =
    QOT_CAND_BAD_SAMPLE | QOT_CAND_BAD_PATH | QOT_CAND_OCCUPIED | QOT_CAND_BAD_STATE | QOT_CAND_BAD_NODE;

template <bool kMove>
__global__ void __launch_bounds__(kCdThreads, 1) lp_candidate_kernel(const __grid_constant__ CdArgs a) {
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = cd_smem().w[w];
  float As[kF], Ad[kF];
  cd_head_prologue(a.prep, As, Ad, tid);
  __syncthreads();
  const float nan = __int_as_float(0x7fc00000);
  const auto flush = [&](int cnt) { cd_flush(w, cnt, a.prep, lane); };
  int zc = 0;                                   // rows staged in this warp's head buffer
  for (int64_t k = static_cast<int64_t>(blockIdx.x) * kCdWarps + w; k < a.K;
       k += static_cast<int64_t>(gridDim.x) * kCdWarps) {
    // ---- validation
    int st = 0;
    const int64_t s = a.sample[k];
    if (s < 0 || s >= a.S) st |= QOT_CAND_BAD_SAMPLE;
    const int64_t jg = kMove ? a.node[k] : -1;            // moved lightpath (state-batch node), -1 = an insertion
    const int64_t p0 = a.link_ptr[k], p1 = a.link_ptr[k + 1];
    const bool tear = kMove && jg >= 0 && p1 == p0;       // a teardown: no new placement, q0 / width / feat unused
    const int c0 = a.q0[k], cw = a.width[k];
    if (cd_bad_route(a, a.cfg.L, p0, p1, tear, cw < 1 || c0 < 0 || static_cast<int64_t>(c0) + cw > a.cfg.Q, lane))
      st |= QOT_CAND_BAD_PATH;
    if (kMove && jg != -1 && !(st & QOT_CAND_BAD_SAMPLE) && (jg < a.node_ptr[s] || jg >= a.node_ptr[s + 1]))
      st |= QOT_CAND_BAD_NODE;
    int64_t n0 = 0;
    int n = 0;
    if (st == 0) st |= cd_sample_nodes(a, s, n0, n) ? 0 : QOT_CAND_BAD_STATE;
    const int jm = kMove && st == 0 && jg >= 0 ? static_cast<int>(jg - n0) : -1;   // sample-local; -1 matches no node
    // ---- new neighbours, with the moved lightpath's channels free; its old neighbours
    if (lane < kCdMaskWords) {
      ws.mask[lane] = 0u;
      if (kMove) ws.omask[lane] = 0u;
    }
    __syncwarp();
    if (st == 0) {
      int sb = cd_scan(a, s, n0, n, p0, p1, c0, cw, ws.mask, [&](int j) { return kMove && j == jm; }, lane);
      if (kMove && jm >= 0 && !cd_old_nbrs(a, n0, n, jm, ws.omask, lane)) sb |= QOT_CAND_BAD_STATE;
      st |= __reduce_or_sync(kFull, sb);
    }
    __syncwarp();
    if (st & kCdFatal) {
      if (lane < QOT_OUT) a.out[k * QOT_OUT + lane] = nan;
      if (lane == 0) {
        a.status[k] = st;
        a.n_impact[k] = 0;
      }
      cd_clear_impact(a, k, 0, a.max_impact, kMove ? a.impact_kind : nullptr, lane, 32);
      continue;
    }
    // ---- neighbours of the new placement ranked ascending: lane t < 8 owns mask word t.  A candidate's impact rows
    // are exactly these; a change's own row takes them from msg and its impact rows are ranked below.
    const unsigned mw = lane < kCdMaskWords ? ws.mask[lane] : 0u;
    int* own = kMove ? ws.msg : ws.nbr;
    const int nn = cd_rank(mw, own, lane);
    if (lane == 0) own[nn] = kCand;                               // the candidate's appended self loop
    cd_xrow(a, ws.cx, [&] { return a.feat[k * 4 + lane]; }, lane);
    __syncwarp();
    const float* xs = a.x + n0 * kF;
    if (kMove && tear) {
      if (lane < QOT_OUT) a.out[k * QOT_OUT + lane] = nan;
    } else {
      zc = cd_row(ws, zc, own, nn + 1, kCand, CdX{xs, ws.cx, kCand, a.lut_col}, As, Ad, a.out + k * QOT_OUT, flush,
                  lane);
    }
    int cnt = nn;
    if (kMove) {                             // impact rows of a change: old and new neighbours
      cnt = cd_rank(mw | (lane < kCdMaskWords ? ws.omask[lane] : 0u), ws.nbr, lane);
      __syncwarp();
    }
    const int MI = a.max_impact;
    if (cnt > MI) st |= QOT_CAND_IMPACT_OVERFLOW;
    const int rows = min(cnt, MI);
    for (int i = 0; i < rows; ++i) {
      const int j = ws.nbr[i];
      const int kind = kMove ? static_cast<int>((ws.omask[j >> 5] >> (j & 31) & 1u) |
                                                (ws.mask[j >> 5] >> (j & 31) & 1u) << 1)
                             : 2;            // bit 0: was a neighbour of the moved lightpath, bit 1: is one now
      float* dst = a.impact_out + (k * MI + i) * QOT_OUT;
      if (lane == 0) {
        a.impact_node[k * MI + i] = n0 + j;
        if (kMove && a.impact_kind) a.impact_kind[k * MI + i] = static_cast<int8_t>(kind);
      }
      const int m = cd_in_row(a, n0, n, j, ws.msg, lane, [&](int d) { return kMove && d == jm; });
      if (m < 0) {
        st |= QOT_CAND_BAD_STATE;
        if (lane < QOT_OUT) dst[lane] = nan;
        __syncwarp();
        continue;
      }
      const int mc = kind >> 1;               // the candidate / moved lightpath is a message of new neighbours only
      if (lane == 0) {
        if (mc) ws.msg[m] = kCand;
        ws.msg[m + mc] = j;
      }
      __syncwarp();
      zc = cd_row(ws, zc, ws.msg, m + mc + 1, j, CdX{xs, ws.cx, j, a.lut_col}, As, Ad, dst, flush, lane);
    }
    cd_clear_impact(a, k, rows, MI, kMove ? a.impact_kind : nullptr, lane, 32);
    if (lane == 0) {
      a.status[k] = st;
      a.n_impact[k] = cnt;
    }
  }
  if (zc) flush(zc);
}

// ------------------------------------------------------------------------------------------------ change sets
// lp_change_set_kernel: persistent, one warp per set of changes to one sample (qot_lightpath_change_sets).  The set's
// removed lightpaths R (the nodes its changes move or tear down) go into a 256-bit mask; each placed change scans its
// path's chan_node rows with R counted as free, its new neighbours into its own 256-bit mask; the placed changes are
// tested pairwise (a shared link and 0 < |df| < threshold: adjacent; a shared channel: a conflict); R's out-runs give
// the old neighbours.  The impact rows are the union of all masks without R, ranked ascending.  Changed lightpath c is
// message source -1 - c (its scaled x row in the warp's table), so a set of one change runs the reconfiguration rows
// with the same message order and values: bit-identical to lp_candidate_kernel<true>.
constexpr int kCsMaxChanges = QOT_SET_MAX_CHANGES;
constexpr int kCsMsgCap = kCdMaxN + kCsMaxChanges + 8;  // in-row (<= kCdMaxN) + changed lightpaths + self loop
constexpr int kCsFatal = kCdFatal | QOT_SET_BAD_SET | QOT_SET_DUPLICATE | QOT_SET_CONFLICT;
static_assert(kCsMaxChanges == 64, "the pairwise matrix and the per-set bit words hold 64 changes");

struct CsWarpSmem {
  unsigned nmask[kCsMaxChanges][kCdMaskWords];  // new-neighbour bits of each change
  float cx[kCsMaxChanges][8];                   // scaled x row of each change
  unsigned long long adj[kCsMaxChanges];        // bit d of row c: changes c and d are adjacent
  int msg[kCsMsgCap];                           // message list of one row
  int st[kCsMaxChanges];                        // status bits of each change
  int jm[kCsMaxChanges];                        // sample-local node each change moves or tears down, -1: none
  unsigned rmask[kCdMaskWords];                 // R: the lightpaths the set moves or tears down
  unsigned char tear[kCsMaxChanges];            // the change is a teardown
  long long k0, n0;                             // the set's first change and its sample's first node
  int nc, n, cnt, any;                          // changes, the sample's nodes, impact rows, OR of the status words
};
struct CsSmem {
  CdSmem cd;                                    // head fragments and the candidate kernel's per-warp state
  CsWarpSmem w[kCdWarps];
};
static_assert(sizeof(CsSmem) + 16 <= 227 * 1024, "lp_change_set_kernel: shared memory over the 227 KB block limit");

// x of a message source: sample-local node j >= 0 of the state, or changed lightpath -1 - j of the set
struct CsX {
  const float* __restrict__ xs;
  const float (*cx)[8];
  int lut, col;
  __device__ __forceinline__ float operator()(int j, int k) const {
    if (k == col) return j == lut ? 1.0f : 0.0f;
    return j < 0 ? cx[-1 - j][k] : __ldg(xs + static_cast<int64_t>(j) * kF + k);
  }
};

struct CsArgs {
  CdArgs c;                                // the reconfiguration arguments; status, n_impact and impact_* are per set
  int64_t G;
  const int64_t* set_ptr;
  float* chg_out;                          // [K,3]
  int32_t* chg_status;                     // [K]
};

__device__ __forceinline__ bool cs_bit(const unsigned* m, int j) { return m[j >> 5] >> (j & 31) & 1u; }

__global__ void __launch_bounds__(kCdThreads, 1) lp_change_set_kernel(const __grid_constant__ CsArgs ca) {
  const CdArgs& a = ca.c;
  CsSmem& sm = *reinterpret_cast<CsSmem*>(cd_smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = sm.cd.w[w];
  CsWarpSmem& xw = sm.w[w];
  float As[kF], Ad[kF];
  cd_head_prologue(a.prep, As, Ad, tid);
  // set_ptr must partition [0, K): non-decreasing from 0 to K.  Otherwise sets could overlap, so none is evaluated:
  // every change and every set gets BAD_SET, each output written by exactly one thread of the grid.
  bool bad_ptr = false;
  for (int64_t g = tid; g <= ca.G; g += kCdThreads) {
    const int64_t v = ca.set_ptr[g];
    bad_ptr |= (g == 0 && v != 0) || (g == ca.G && v != a.K) || (g < ca.G && ca.set_ptr[g + 1] < v);
  }
  bad_ptr = __syncthreads_or(bad_ptr);
  const float nan = __int_as_float(0x7fc00000);
  if (bad_ptr) {
    const int64_t gt = static_cast<int64_t>(blockIdx.x) * kCdThreads + tid;
    const int64_t gs = static_cast<int64_t>(gridDim.x) * kCdThreads;
    for (int64_t k = gt; k < a.K; k += gs) {
      ca.chg_status[k] = QOT_SET_BAD_SET;
      for (int o = 0; o < QOT_OUT; ++o) ca.chg_out[k * QOT_OUT + o] = nan;
    }
    for (int64_t g = gt; g < ca.G; g += gs) {
      a.status[g] = QOT_SET_BAD_SET;
      a.n_impact[g] = 0;
      cd_clear_impact(a, g, 0, a.max_impact, a.impact_kind, 0, 1);
    }
    return;
  }
  const auto flush = [&](int cnt) { cd_flush(w, cnt, a.prep, lane); };
  int zc = 0;                                       // rows staged in this warp's head buffer
  for (int64_t g = static_cast<int64_t>(blockIdx.x) * kCdWarps + w; g < ca.G;
       g += static_cast<int64_t>(gridDim.x) * kCdWarps) {
    const int64_t k0 = ca.set_ptr[g], nk = ca.set_ptr[g + 1] - k0;
    const int nc = nk > kCsMaxChanges ? 0 : static_cast<int>(nk);   // a set over the limit is not examined
    const int64_t s = nc ? a.sample[k0] : -1;
    int64_t n0 = 0;
    int n = 0;
    const bool state_ok = s >= 0 && s < a.S && cd_sample_nodes(a, s, n0, n);
    if (lane < kCdMaskWords) {
      xw.rmask[lane] = 0u;
      ws.mask[lane] = 0u;
      ws.omask[lane] = 0u;
    }
    __syncwarp();
    // ---- each change: the reconfiguration checks, the set's sample, R, the scaled x row
    for (int c = 0; c < nc; ++c) {
      const int64_t k = k0 + c;
      int st = 0;
      const int64_t sk = a.sample[k];
      if (sk < 0 || sk >= a.S) st |= QOT_CAND_BAD_SAMPLE;
      if (sk != s) st |= QOT_SET_BAD_SET;
      const int64_t jg = a.node[k];
      const int64_t p0 = a.link_ptr[k], p1 = a.link_ptr[k + 1];
      const bool tear = jg >= 0 && p1 == p0;        // a teardown: no new placement, q0 / width / feat unused
      const int c0 = a.q0[k], cw = a.width[k];
      if (cd_bad_route(a, a.cfg.L, p0, p1, tear, cw < 1 || c0 < 0 || static_cast<int64_t>(c0) + cw > a.cfg.Q, lane))
        st |= QOT_CAND_BAD_PATH;
      if (jg != -1 && !(st & QOT_CAND_BAD_SAMPLE) && (jg < a.node_ptr[sk] || jg >= a.node_ptr[sk + 1]))
        st |= QOT_CAND_BAD_NODE;
      if (st == 0 && !state_ok) st |= QOT_CAND_BAD_STATE;
      const int jm = st == 0 && jg >= 0 ? static_cast<int>(jg - n0) : -1;
      if (lane == 0) {
        if (jm >= 0) {
          if (cs_bit(xw.rmask, jm)) st |= QOT_SET_DUPLICATE;
          xw.rmask[jm >> 5] |= 1u << (jm & 31);
        }
        xw.st[c] = st;
        xw.jm[c] = jm;
        xw.tear[c] = tear;
      }
      if (lane < kCdMaskWords) xw.nmask[c][lane] = 0u;
      cd_xrow(a, xw.cx[c], [&] { return a.feat[k * 4 + lane]; }, lane);
      __syncwarp();
    }
    if (lane == 0)                                  // every change removing a lightpath removed twice
      for (int c = 1; c < nc; ++c)
        if (xw.st[c] & QOT_SET_DUPLICATE)
          for (int d = 0; d < c; ++d)
            if (xw.jm[d] == xw.jm[c]) xw.st[d] |= QOT_SET_DUPLICATE;
    __syncwarp();
    int any = nk > kCsMaxChanges ? QOT_SET_BAD_SET : 0;
    for (int c = 0; c < nc; ++c) any |= xw.st[c];
    if (!(any & kCsFatal)) {
      // ---- new neighbours of each placed change; R's channels are free and R is no neighbour
      for (int c = 0; c < nc; ++c) {
        if (xw.tear[c]) continue;
        const int64_t k = k0 + c;
        const int sb = cd_scan(a, s, n0, n, a.link_ptr[k], a.link_ptr[k + 1], a.q0[k], a.width[k], xw.nmask[c],
                               [&](int j) { return cs_bit(xw.rmask, j); }, lane);
        const int sw = __reduce_or_sync(kFull, sb);
        if (lane == 0) xw.st[c] |= sw;
      }
      // ---- old neighbours: the destinations of R's out-runs, self loops dropped
      for (int c = 0; c < nc; ++c) {
        const int jm = xw.jm[c];
        if (jm < 0) continue;
        if (__any_sync(kFull, !cd_old_nbrs(a, n0, n, jm, ws.omask, lane)) && lane == 0) xw.st[c] |= QOT_CAND_BAD_STATE;
      }
      // ---- pairs of placed changes, one lane per pair: a shared link and a shared slot is a conflict, a shared link
      // and cd_df_hit between the two slot ranges an edge
      for (int c = lane; c < nc; c += 32) xw.adj[c] = 0ull;
      __syncwarp();
      for (int pr = lane; pr < nc * nc; pr += 32) {
        const int c = pr / nc, d = pr - c * nc;
        if (d <= c || xw.tear[c] || xw.tear[d]) continue;
        const int64_t kc = k0 + c, kd = k0 + d;
        bool share = false;
        for (int64_t e = a.link_ptr[kc]; e < a.link_ptr[kc + 1] && !share; ++e)
          for (int64_t f = a.link_ptr[kd]; f < a.link_ptr[kd + 1] && !share; ++f) share = a.links[e] == a.links[f];
        if (!share) continue;
        const int c0 = a.q0[kc], cw = a.width[kc], d0 = a.q0[kd], dw = a.width[kd];
        if (c0 < d0 + dw && d0 < c0 + cw) {
          atomicOr(&xw.st[c], QOT_SET_CONFLICT);
          atomicOr(&xw.st[d], QOT_SET_CONFLICT);
          continue;
        }
        bool hit = false;
        for (int qd = d0; qd < d0 + dw && !hit; ++qd)
          hit = cd_df_hit(a.freqs, a.freqs[qd], c0, cw, a.cfg.freq_threshold);
        if (hit) {
          atomicOr(&xw.adj[c], 1ull << d);
          atomicOr(&xw.adj[d], 1ull << c);
        }
      }
      __syncwarp();
      any = 0;
      for (int c = 0; c < nc; ++c) any |= xw.st[c];
    }
    // ---- impact rows: every lightpath outside R adjacent to a changed one before or after, ascending; their in-rows
    // are checked before any row is emitted, so that a bad state leaves the whole set NaN
    int cnt = 0;
    if (!(any & kCsFatal)) {
      if (lane < kCdMaskWords) {
        unsigned nw = 0u;
        for (int c = 0; c < nc; ++c) nw |= xw.nmask[c][lane];
        ws.mask[lane] = nw;
        ws.omask[lane] &= ~xw.rmask[lane];
      }
      __syncwarp();
      const unsigned uw = lane < kCdMaskWords ? ws.mask[lane] | ws.omask[lane] : 0u;
      cnt = cd_rank(uw, ws.nbr, lane);
      __syncwarp();
      bool bad = false;
      for (int i = 0; i < min(cnt, a.max_impact) && !bad; ++i)
        bad = cd_in_row<false>(a, n0, n, ws.nbr[i], nullptr, lane) < 0;
      if (bad) {
        if (lane == 0) xw.st[0] |= QOT_CAND_BAD_STATE;
        any |= QOT_CAND_BAD_STATE;
      }
      if (cnt > a.max_impact && lane == 0)
        for (int c = 0; c < nc; ++c) xw.st[c] |= QOT_CAND_IMPACT_OVERFLOW;
      if (cnt > a.max_impact) any |= QOT_CAND_IMPACT_OVERFLOW;
      __syncwarp();
    }
    if (any & kCsFatal) {                           // a partial joint answer is meaningless: the whole set is NaN
      for (int64_t k = k0 + lane; k < k0 + nk; k += 32) {
        ca.chg_status[k] = nc ? xw.st[k - k0] : QOT_SET_BAD_SET;
        for (int o = 0; o < QOT_OUT; ++o) ca.chg_out[k * QOT_OUT + o] = nan;
      }
      if (lane == 0) {
        a.status[g] = any;
        a.n_impact[g] = 0;
      }
      cd_clear_impact(a, g, 0, a.max_impact, a.impact_kind, lane, 32);
      __syncwarp();
      continue;
    }
    // ---- the rows, one attention call site: the changes in set order (new neighbours ascending, the adjacent
    // changes in set order, the self loop), then the impact rows (the state in-row without R and the self loop, the
    // adjacent changes in set order, the self loop).  The set's scalars live in shared memory across the rows.
    if (lane == 0) {
      xw.k0 = k0;
      xw.n0 = n0;
      xw.nc = nc;
      xw.n = n;
      xw.cnt = cnt;
      xw.any = any;
    }
    __syncwarp();
    for (int r = 0; r < nc + min(cnt, a.max_impact); ++r) {
      const int64_t n0r = xw.n0;
      const int ncr = xw.nc;
      int m = 0, q;
      float* dst;
      if (r < ncr) {                                // the row of change c = r
        dst = ca.chg_out + (xw.k0 + r) * QOT_OUT;
        if (xw.tear[r]) {
          if (lane < QOT_OUT) dst[lane] = nan;
          continue;
        }
        m = cd_rank(lane < kCdMaskWords ? xw.nmask[r][lane] : 0u, xw.msg, lane);
        if (lane == 0) {
          for (unsigned long long b = xw.adj[r]; b; b &= b - 1) xw.msg[m++] = -(__ffsll(static_cast<long long>(b)));
          xw.msg[m++] = -1 - r;
        }
        m = __shfl_sync(kFull, m, 0);
        q = -1 - r;
      } else {                                      // impact row i = r - nc (its in-row was checked above)
        const int i = r - ncr, j = ws.nbr[i];
        const int kind = static_cast<int>(cs_bit(ws.omask, j)) | static_cast<int>(cs_bit(ws.mask, j)) << 1;
        if (lane == 0) {
          a.impact_node[g * a.max_impact + i] = n0r + j;
          if (a.impact_kind) a.impact_kind[g * a.max_impact + i] = static_cast<int8_t>(kind);
        }
        m = cd_in_row(a, n0r, xw.n, j, xw.msg, lane, [&](int d) { return cs_bit(xw.rmask, d); });
        if (kind >> 1)
          for (int cb = 0; cb < ncr; cb += 32) {
            const int c = cb + lane;
            const bool hit = c < ncr && !xw.tear[c] && cs_bit(xw.nmask[c], j);
            const unsigned ball = __ballot_sync(kFull, hit);
            if (hit) xw.msg[m + __popc(ball & ((1u << lane) - 1u))] = -1 - c;
            m += __popc(ball);
          }
        if (lane == 0) xw.msg[m] = j;
        ++m;
        q = j;
        dst = a.impact_out + (g * a.max_impact + i) * QOT_OUT;
      }
      __syncwarp();
      zc = cd_row(ws, zc, xw.msg, m, q, CsX{a.x + n0r * kF, xw.cx, q, a.lut_col}, As, Ad, dst, flush, lane);
    }
    cd_clear_impact(a, g, min(xw.cnt, a.max_impact), a.max_impact, a.impact_kind, lane, 32);
    for (int c = lane; c < xw.nc; c += 32) ca.chg_status[xw.k0 + c] = xw.st[c];
    if (lane == 0) {
      a.status[g] = xw.any;
      a.n_impact[g] = xw.cnt;
    }
    __syncwarp();
  }
  if (zc) flush(zc);
}

// ------------------------------------------------------------------------------------------------ placements
// lp_placement_kernel: persistent, one warp per demand (qot_lightpath_placements).  A demand offers up to 32 options
// (a route, a width, the channel features); a placement is an option with a start slot q0 whose channels are free on
// every link of the route, and its rows are by definition the candidate kernel's rows for that candidate (freq =
// float32(freqs[q0])).  Per option the warp reads each chan_node row of the route once, coalesced: the ballots give the
// occupied bitmap (lane t owns slots [32t, 32t + 32), Q <= 1024) and the occupied channels of known lightpaths are
// collected as (slot, node) entries.  The free starts for the option's width come from log2(width) AND-shift steps
// of the free bitmap, words carried across lanes by shuffles.  Each free start's neighbour mask is the candidate
// kernel's fp64 0 < |df| < threshold test over the collected entries (over the chan_node rows again when the route
// holds more than kPlEntCap of them), ranked as the candidate kernel ranks it.  Own rows (and, with a bound, every
// impact row) go 16 at a time through the head; the staged outputs fold into the placement's margin (an ordered
// integer key, so min and max are exact and order-free) and, once its last row is out, into the demand's running best
// (policy key << 32 | ~(option << 10 | q0): the lower index wins a tie).  The winner is evaluated again at the end of
// the demand for its first max_impact impact rows.
constexpr int kPlMaxOptions = QOT_PLACE_MAX_OPTIONS;
constexpr int kPlMaxQ = QOT_PLACE_MAX_SLOTS;
constexpr int kPlEntCap = 768;                     // (slot, node) entries of one route; more: scan chan_node again
constexpr int kPlRing = 32;                        // placements with rows in the head buffer: at most 17
constexpr int kPlFatal = QOT_CAND_BAD_SAMPLE | QOT_CAND_BAD_PATH | QOT_CAND_BAD_STATE;
static_assert(kPlMaxQ == 32 * 32, "one 32-bit free word per lane");
static_assert(kPlMaxOptions <= 32 && kPlMaxQ <= 1024, "option << 10 | q0 fits the low key word");

struct PlPending {                           // a placement whose rows are in flight
  float own[3];
  unsigned mkey;                             // min of the row margins' ordered keys (0: a NaN margin)
  int left, p, q0;                           // rows not yet folded, option (global), start slot
};
struct PlWarpSmem {
  int ent[kPlEntCap];                        // the route's occupied channels of known lightpaths: slot << 8 | node
  PlPending ring[kPlRing];
  float rout[16][4];                         // outputs of the staged rows of the search
  long long rnode[16];                       // bound index of a staged impact row, -1: an own row
  int rtag[16];                              // ring slot of a staged row, -1: a winner's row (written out directly)
  unsigned long long key;                    // the demand's running best (0: none feasible yet)
  float best[4];                             // its own row and margin
  int n_free, n_feas;
};
struct PlSmem {
  CdSmem cd;                                 // head fragments and the candidate kernel's per-warp state
  PlWarpSmem w[kCdWarps];
};
static_assert(sizeof(PlSmem) + 16 <= 227 * 1024, "lp_placement_kernel: shared memory over the 227 KB block limit");

struct PlArgs {
  CdArgs c;                                // state, links, width, prep, max_impact, status / n_impact / impact_*
  int64_t P;                               // options
  const int64_t* opt_ptr;                  // [D+1]
  const float* own_bound;                  // [P]
  const float* bound;                      // [N] or null
  int metric, maximize, policy;
  int32_t* option;                         // [D]
  int32_t* q0;                             // [D]
  float* margin;                           // [D]
  int32_t* n_free;
  int32_t* n_feasible;
  float* all_out;                          // [P,Q,3] or null
  float* all_margin;                       // [P,Q] or null
};

// float -> unsigned, monotone (-0 counts as +0); NaN -> 0, below every number
__device__ __forceinline__ unsigned pl_okey(float f) {
  if (f != f) return 0u;
  const unsigned u = __float_as_uint(__fadd_rn(f, 0.0f));
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float pl_unkey(unsigned k) {
  if (k == 0u) return __int_as_float(0x7fc00000);
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// bit i of lane t's word of the result = slot 32t + i + k of x (slots past the last word read as 0, occupied)
__device__ __forceinline__ unsigned pl_shr(unsigned x, int k, int lane) {
  const int d = k >> 5, b = k & 31;
  unsigned lo = __shfl_down_sync(kFull, x, d), hi = __shfl_down_sync(kFull, x, d + 1);
  if (lane + d > 31) lo = 0u;
  if (lane + d + 1 > 31) hi = 0u;
  return b ? (lo >> b) | (hi << (32 - b)) : lo;
}

// the free starts for width cw (lane t: word t): AND of the free bits over [q0, q0 + cw), in log2(cw) shift steps
__device__ __forceinline__ unsigned pl_free_starts(unsigned occ, int Q, int cw, int lane) {
  const int tail = Q - 32 * lane;
  const unsigned valid = tail >= 32 ? 0xffffffffu : tail > 0 ? (1u << tail) - 1u : 0u;
  unsigned run = ~occ & valid;
  for (int have = 1; have < cw;) {
    const int step = min(have, cw - have);
    run &= pl_shr(run, step, lane);
    have += step;
  }
  return run;
}

// the neighbour bits of placement [q0, q0 + cw) from a route's entries: cd_df_hit against each entry's slot
__device__ __forceinline__ void pl_ent_mask(const CdArgs& a, const int* ent, int ne, int q0, int cw, unsigned* mask,
                                            int lane) {
  for (int i = lane; i < ne; i += 32) {
    const int en = ent[i], q = en >> 8, j = en & 255;
    if (cd_df_hit(a.freqs, a.freqs[q], q0, cw, a.cfg.freq_threshold)) atomicOr(&mask[j >> 5], 1u << (j & 31));
  }
}

// the staged rows' outputs, in staging order, into their placements' margins; a placement whose last row is out goes
// into the demand's count and running best, and into all_out / all_margin.  Lane 0.
__device__ __noinline__ void pl_fold(const PlArgs& a, PlWarpSmem& pw, int cnt, int64_t o0) {
  const int Q = a.c.cfg.Q;
  for (int r = 0; r < cnt; ++r) {
    const int t = pw.rtag[r];
    if (t < 0) continue;
    PlPending& pp = pw.ring[t];
    const float v = pw.rout[r][a.metric];
    const long long nd = pw.rnode[r];
    const float b = nd < 0 ? a.own_bound[pp.p] : a.bound[nd];
    const unsigned k = pl_okey(a.maximize ? __fsub_rn(v, b) : __fsub_rn(b, v));
    pp.mkey = min(pp.mkey, k);
    if (nd < 0)
      for (int o = 0; o < QOT_OUT; ++o) pp.own[o] = pw.rout[r][o];
    if (--pp.left) continue;
    const float mg = pl_unkey(pp.mkey);
    const int64_t at = static_cast<int64_t>(pp.p) * Q + pp.q0;
    if (a.all_out) {
      for (int o = 0; o < QOT_OUT; ++o) a.all_out[at * QOT_OUT + o] = pp.own[o];
      a.all_margin[at] = mg;
    }
    if (pp.mkey < 0x80000000u) continue;               // margin < 0 or NaN: not feasible
    ++pw.n_feas;
    const float ov = pp.own[a.metric];
    const unsigned hi = a.policy == QOT_PLACE_FIRST_FIT ? 0u
                        : a.policy == QOT_PLACE_BEST_QOT ? pl_okey(a.maximize ? ov : -ov)
                                                         : pp.mkey;
    const unsigned idx = static_cast<unsigned>(pp.p - o0) << 10 | static_cast<unsigned>(pp.q0);
    const unsigned long long key = static_cast<unsigned long long>(hi) << 32 | (0xffffffffu - idx);
    if (key > pw.key) {
      pw.key = key;
      for (int o = 0; o < QOT_OUT; ++o) pw.best[o] = pp.own[o];
      pw.best[3] = mg;
    }
  }
}

__device__ __noinline__ void pl_flush(const PlArgs& a, PlWarpSmem& pw, int w, int cnt, int64_t o0, int lane) {
  cd_flush(w, cnt, a.c.prep, lane);
  if (lane == 0) pl_fold(a, pw, cnt, o0);
  __syncwarp();
}

__global__ void __launch_bounds__(kCdThreads, 1) lp_placement_kernel(const __grid_constant__ PlArgs pa) {
  const CdArgs& a = pa.c;
  PlSmem& sm = *reinterpret_cast<PlSmem*>(cd_smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = sm.cd.w[w];
  PlWarpSmem& pw = sm.w[w];
  float As[kF], Ad[kF];
  cd_head_prologue(a.prep, As, Ad, tid);
  __syncthreads();
  const float nan = __int_as_float(0x7fc00000);
  int zc = 0;                                             // rows staged in this warp's head buffer
  for (int64_t d = static_cast<int64_t>(blockIdx.x) * kCdWarps + w; d < a.K;
       d += static_cast<int64_t>(gridDim.x) * kCdWarps) {
    const int L = a.cfg.L, Q = a.cfg.Q;
    // ---- validation: the sample, the option range, every option's route and width, the state offsets
    int st = 0;
    const int64_t s = a.sample[d];
    if (s < 0 || s >= a.S) st |= QOT_CAND_BAD_SAMPLE;
    const int64_t o0 = pa.opt_ptr[d], o1 = pa.opt_ptr[d + 1];
    const bool opts_ok = o0 >= 0 && o1 > o0 && o1 <= pa.P && o1 - o0 <= kPlMaxOptions;
    bool badp = !opts_ok;
    if (opts_ok)
      for (int64_t po = o0; po < o1 && !badp; ++po) {
        const int cw = a.width[po];
        badp = cd_bad_route(a, L, a.link_ptr[po], a.link_ptr[po + 1], false, cw < 1 || cw > Q, lane);
      }
    if (badp) st |= QOT_CAND_BAD_PATH;
    int64_t n0 = 0;
    int n = 0;
    if (st == 0) st |= cd_sample_nodes(a, s, n0, n) ? 0 : QOT_CAND_BAD_STATE;
    if (lane == 0) {
      pw.key = 0ull;
      pw.n_free = pw.n_feas = 0;
    }
    __syncwarp();
    const float* xs = a.x + n0 * kF;
    // a row of the search (ring slot `tag`, bound index `node`, -1 for an own row; its outputs staged for pl_fold) or
    // of the winner (tag -1, its outputs to dst)
    const auto row = [&](const int* msg, int M, int q, float* dst, int tag, long long node) {
      if (lane == 0) {
        pw.rtag[zc] = tag;
        pw.rnode[zc] = node;
      }
      zc = cd_row(ws, zc, msg, M, q, CdX{xs, ws.cx, q, a.lut_col}, As, Ad, dst ? dst : pw.rout[zc],
                  [&](int cnt) { pl_flush(pa, pw, w, cnt, o0, lane); }, lane);
    };
    int seq = 0;                                          // placements of this demand, for the ring slots
    for (int64_t po = o0; st == 0 && po < o1; ++po) {
      const int64_t p0 = a.link_ptr[po], p1 = a.link_ptr[po + 1];
      const int cw = a.width[po];
      // ---- the route's occupied bitmap (lane t: word t) and its channels of known lightpaths, one read per row
      unsigned occ = 0u;
      int ne = 0;
      bool bad = false;
      for (int64_t e = p0; e < p1; ++e) {
        const int32_t* __restrict__ crow = a.chan_node + (s * L + a.links[e]) * Q;
        for (int qb = 0; qb < Q; qb += 32) {
          const int q = qb + lane;
          const int32_t v = q < Q ? crow[q] : -1;
          const unsigned ob = __ballot_sync(kFull, v != -1);
          if (lane == qb >> 5) occ |= ob;
          const int64_t j = static_cast<int64_t>(v) - n0;
          const bool known = v >= 0 && j >= 0 && j < n;
          bad |= v >= 0 && !known;
          const bool keep = known;                        // every link's channels of known lightpaths
          const unsigned kb = __ballot_sync(kFull, keep);
          const int at = ne + __popc(kb & ((1u << lane) - 1u));
          if (keep && at < kPlEntCap) pw.ent[at] = q << 8 | static_cast<int>(j);
          ne += __popc(kb);
        }
      }
      if (__any_sync(kFull, bad)) {
        st |= QOT_CAND_BAD_STATE;
        break;
      }
      __syncwarp();
      // ---- free starts for width cw: AND of the free bits over [q0, q0 + cw), in log2(cw) shift steps
      const unsigned run = pl_free_starts(occ, Q, cw, lane);
      if (pa.all_out)                                     // NaN at every start that is not free
        for (int wd = 0; wd < 32 && 32 * wd < Q; ++wd) {
          const unsigned bits = __shfl_sync(kFull, run, wd);
          const int q = 32 * wd + lane;
          if (q >= Q || (bits >> lane & 1u)) continue;
          const int64_t at = po * Q + q;
          pa.all_margin[at] = nan;
          for (int o = 0; o < QOT_OUT; ++o) pa.all_out[at * QOT_OUT + o] = nan;
        }
      // ---- every free start in ascending order; its neighbours from the collected entries (the placement's own
      // channels are free), or from the chan_node rows again when the route held more than kPlEntCap of them
      for (int wd = 0; wd < 32 && 32 * wd < Q; ++wd) {
        for (unsigned bits = __shfl_sync(kFull, run, wd); bits; bits &= bits - 1u) {
          const int q0 = 32 * wd + __ffs(bits) - 1;
          if (lane < kCdMaskWords) ws.mask[lane] = 0u;
          __syncwarp();
          if (ne <= kPlEntCap) {
            pl_ent_mask(a, pw.ent, ne, q0, cw, ws.mask, lane);
          } else {
            cd_scan(a, s, n0, n, p0, p1, q0, cw, ws.mask, CdNone(), lane);
          }
          __syncwarp();
          const int nn = cd_rank(lane < kCdMaskWords ? ws.mask[lane] : 0u, ws.nbr, lane);
          cd_xrow(a, ws.cx, [&] { return lane == 0 ? static_cast<float>(a.freqs[q0]) : a.feat[po * 3 + lane - 1]; },
                  lane);
          const int slot = seq++ & (kPlRing - 1);
          const int nimp = pa.bound ? nn : 0;             // impact rows count against a bound, all of them
          if (lane == 0) {
            ws.nbr[nn] = kCand;
            PlPending& pp = pw.ring[slot];
            pp.mkey = 0xffffffffu;
            pp.left = 1 + nimp;
            pp.p = static_cast<int>(po);
            pp.q0 = q0;
            ++pw.n_free;
          }
          __syncwarp();
          row(ws.nbr, nn + 1, kCand, nullptr, slot, -1);
          for (int i = 0; i < nimp; ++i) {                // whatever max_impact is
            const int j = ws.nbr[i];
            const int m = cd_in_row(a, n0, n, j, ws.msg, lane);
            if (m < 0) {
              st |= QOT_CAND_BAD_STATE;
              break;
            }
            if (lane == 0) {
              ws.msg[m] = kCand;
              ws.msg[m + 1] = j;
            }
            __syncwarp();
            row(ws.msg, m + 2, j, nullptr, slot, n0 + j);
          }
          if (st) break;
        }
        if (st) break;
      }
    }
    // ---- every placement of the demand folded: the winner
    if (zc) {
      pl_flush(pa, pw, w, zc, o0, lane);
      zc = 0;
    }
    const int MI = a.max_impact;
    const unsigned long long key = pw.key;
    int cnt = 0, rows = 0, bp = -1, bq = -1;
    if (st == 0 && key) {
      const unsigned idx = 0xffffffffu - static_cast<unsigned>(key);
      bp = static_cast<int>(idx >> 10);
      bq = static_cast<int>(idx & 1023u);
      const int64_t po = o0 + bp;
      if (lane < kCdMaskWords) ws.mask[lane] = 0u;
      __syncwarp();
      cd_scan(a, s, n0, n, a.link_ptr[po], a.link_ptr[po + 1], bq, a.width[po], ws.mask, CdNone(), lane);
      __syncwarp();
      cnt = cd_rank(lane < kCdMaskWords ? ws.mask[lane] : 0u, ws.nbr, lane);
      __syncwarp();
      rows = min(cnt, MI);
      bool bad = false;                                   // in-rows checked before any row is written
      for (int i = 0; i < rows && !bad; ++i) bad = cd_in_row<false>(a, n0, n, ws.nbr[i], nullptr, lane) < 0;
      if (bad) st |= QOT_CAND_BAD_STATE;
      cd_xrow(a, ws.cx, [&] { return lane == 0 ? static_cast<float>(a.freqs[bq]) : a.feat[po * 3 + lane - 1]; },
              lane);
      __syncwarp();
    }
    if (st & kPlFatal) {
      if (lane < QOT_OUT) a.out[d * QOT_OUT + lane] = nan;
      if (lane == 0) {
        a.status[d] = st;
        a.n_impact[d] = 0;
        pa.option[d] = pa.q0[d] = -1;
        pa.margin[d] = nan;
        pa.n_free[d] = pa.n_feasible[d] = 0;
      }
      cd_clear_impact(a, d, 0, MI, nullptr, lane, 32);
      if (pa.all_out && opts_ok)
        for (int64_t i = o0 * Q + lane; i < o1 * Q; i += 32) {
          pa.all_margin[i] = nan;
          for (int o = 0; o < QOT_OUT; ++o) pa.all_out[i * QOT_OUT + o] = nan;
        }
      __syncwarp();
      continue;
    }
    // ---- the winner's impact rows (their in-rows were checked above)
    for (int i = 0; i < rows; ++i) {
      const int j = ws.nbr[i];
      if (lane == 0) a.impact_node[d * MI + i] = n0 + j;
      const int m = cd_in_row(a, n0, n, j, ws.msg, lane);
      if (lane == 0) {
        ws.msg[m] = kCand;
        ws.msg[m + 1] = j;
      }
      __syncwarp();
      row(ws.msg, m + 2, j, a.impact_out + (d * MI + i) * QOT_OUT, -1, -1);
    }
    cd_clear_impact(a, d, rows, MI, nullptr, lane, 32);
    if (lane < QOT_OUT) a.out[d * QOT_OUT + lane] = key ? pw.best[lane] : nan;
    if (lane == 0) {
      a.status[d] = st | (cnt > MI ? QOT_CAND_IMPACT_OVERFLOW : 0);
      a.n_impact[d] = cnt;
      pa.option[d] = bp;
      pa.q0[d] = bq;
      pa.margin[d] = key ? pw.best[3] : nan;
      pa.n_free[d] = pw.n_free;
      pa.n_feasible[d] = pw.n_feas;
    }
    __syncwarp();
  }
  if (zc) pl_flush(pa, pw, w, zc, 0, lane);
}

// ------------------------------------------------------------------------------------------------ provisioning
// lp_provision_kernel: persistent, one block per sample (qot_lightpath_provision).  The sample's demands are taken in
// order, each placed as lp_placement_kernel places it against the state with every earlier accepted demand of the
// sample written in.  The block holds that state as a dense graph in node-rank order: a 256 x 256-bit adjacency from
// the out-runs (self loops dropped), the x rows, the conn_ids and each node's first channel (link * Q + slot: the
// graph builder orders nodes by it).  Accepted channels go into chan_work, the entry point's copy of chan_node, which
// the block reads through L2 (__ldcg) because it writes it; a channel there holds n0 + the node's stable id (state
// node j: j; the c-th accepted demand: n + c) and s2r maps a stable id to its rank.
//   per demand and option: warp 0 scans the route into the free-start words (pl_free_starts) and (slot << 8 | rank)
//     entries; the free placements are dealt round-robin to the warps, each evaluating its placements as the placement
//     kernel does (own row: the neighbours by rank, then the self loop; impact row of rank r: r's adjacency row by
//     rank, the placement, the self loop) and folding them with pl_fold into its own best key and counts;
//   the block takes the largest key (unique: its low word is the placement's index) and the summed counts, so the
//     choice does not depend on which warp evaluated what; warp 0 writes the winner's impact rows;
//   an accepted demand is inserted at the rank its first channel (min route link, q0) gives it: every row's bits from
//     that rank up move one place, its row and column go in, its channels into chan_work, its own_bound into
//     bound_work (the bound of its impact rows from then on).
// Message order and values are then those of lp_placement_kernel on the rebuilt state: bit-identical.
//
// Releases (qot_lightpath_traffic; none for qot_lightpath_provision): before demand d the block applies the sample's
// releases with before <= d, after its last demand the rest.  A release finds its lightpath's rank by conn_id
// (conn_id[demand] for a release by demand, written earlier by this block), evaluates the rows of its neighbours
// (adj[R]'s bits by rank, each its adjacency row by rank with bit R cleared, then its self loop: the KIND_LOST rows of
// lp_candidate_kernel<true> for the teardown) and folds their margins against bound_work, then pv_release takes the
// lightpath out: its channels in chan_work become -1, the highest stable id takes over its freed id (stable ids stay
// dense in [0, n_tot), which the j < n_tot checks of the route scans rely on), and rank R leaves the graph, every row's
// bits above R moving down one place.  top is not lowered, so conn_ids are never reused within a call.
//
// The kernel is templated on kReleases: the release path takes the kernel from 28 to 148 bytes of spill loads, and a
// launch without releases (qot_lightpath_provision, and qot_lightpath_traffic with R = 0) runs the code it ran before
// releases existed.
struct PvSmem {
  CdSmem cd;                                 // head fragments and the candidate kernel's per-warp state
  PlWarpSmem w[kCdWarps];                    // the placement kernel's per-warp search state
  unsigned adj[kCdMaxN][kCdMaskWords];       // the sample's graph by rank, self loops dropped
  float x[kCdMaxN][kF];                      // x rows by rank
  long long conn[kCdMaxN];                   // conn_id by rank
  int key[kCdMaxN];                          // first channel (link * Q + slot) by rank
  short r2s[kCdMaxN], s2r[kCdMaxN];          // rank <-> stable id
  int ent[kPlEntCap];                        // the option's channels of known lightpaths: slot << 8 | rank
  unsigned run[32];                          // the option's free-start words
  unsigned wmask[kCdMaskWords];              // the winner's neighbours by rank
  float best[4];                             // the winner's own row and margin
  unsigned long long key_best, n_valid;
  long long top;                             // the sample's largest conn_id (at least 0)
  int n_tot, n_chan, ne, rbad, st, n_free, n_feas, acc, c_key;
  long long c_po;
  int c_q0;
  unsigned long long n_rvalid;               // releases with a sample in [0, S), counted by the grouping check
  long long r_conn;                          // the release's conn_id
  int r_st, r_rank;                          // its status so far and its rank (-1: not in the sample)
  unsigned r_mkey;                           // min of its neighbour rows' margin keys
};
static_assert(sizeof(PvSmem) + 16 <= 227 * 1024, "lp_provision_kernel: shared memory over the 227 KB block limit");
static_assert(kCdThreads >= kCdMaxN + 1, "one thread per rank, and one more for the inserted row");

struct PvArgs {
  PlArgs p;                                // p.c.chan_node = chan_work, p.c.impact_node = impact_conn, p.bound =
                                           // bound_work (or null)
  const int64_t* order;                    // [D]: the demands grouped by sample, ascending within a sample
  const int64_t* sample_ptr;               // [S+1]: sample s's demands are order[sample_ptr[s], sample_ptr[s+1])
  const int64_t* conn_ids;                 // [N]
  const float* bound;                      // [N] or null
  int32_t* chan_work;                      // [S, L, Q]
  float* bound_work;                       // [S, kCdMaxN] by stable id, or null
  int64_t* conn_id;                        // [D]
  qot_lp_releases_t rel;                   // R = 0: none (qot_lightpath_provision)
  const int64_t* rel_order;                // [R]: the releases grouped by sample, by (before, k) within a sample
  const int64_t* rel_ptr;                  // [S+1], or null with R = 0
  int32_t* rel_status;                     // [R]
  int64_t* rel_conn_id;                    // [R]
  int32_t* rel_n_impact;                   // [R]
  int64_t* rel_impact_conn;                // [R, max_impact]
  float* rel_impact_out;                   // [R, max_impact, 3]
  float* rel_margin;                       // [R]
};

// x of a message source: rank j of the block's graph or the placement (kCand)
struct PvX {
  const float (*x)[kF];
  const float* cx;
  int lut, col;
  __device__ __forceinline__ float operator()(int j, int k) const {
    if (k == col) return j == lut ? 1.0f : 0.0f;
    return j == kCand ? cx[k] : x[j][k];
  }
};

// the empty result of demand d with status st (option = q0 = -1, NaN rows, zero counts, conn_id -1), written by
// threads t, t + stride, ...
__device__ void pv_empty(const PvArgs& va, int64_t d, int st, int t, int stride) {
  const PlArgs& pa = va.p;
  const CdArgs& a = pa.c;
  const float nan = __int_as_float(0x7fc00000);
  if (t == 0) {
    a.status[d] = st;
    a.n_impact[d] = 0;
    pa.option[d] = pa.q0[d] = -1;
    pa.margin[d] = nan;
    pa.n_free[d] = pa.n_feasible[d] = 0;
    va.conn_id[d] = -1;
  }
  for (int o = t; o < QOT_OUT; o += stride) a.out[d * QOT_OUT + o] = nan;
  cd_clear_impact(a, d, 0, a.max_impact, nullptr, t, stride);
}

// the empty result of release k with status st (conn_id -1, n_impact 0, margin NaN) and its impact rows from `from`
// on (-1 / NaN), written by threads t, t + stride, ...
__device__ void pv_rel_empty(const PvArgs& va, int64_t k, int st, int from, int t, int stride) {
  const int MI = va.p.c.max_impact;
  if (t == 0 && from == 0) {
    va.rel_status[k] = st;
    va.rel_conn_id[k] = -1;
    va.rel_n_impact[k] = 0;
    va.rel_margin[k] = __int_as_float(0x7fc00000);
  }
  for (int i = from + t; i < MI; i += stride) va.rel_impact_conn[k * MI + i] = -1;
  for (int i = from * QOT_OUT + t; i < MI * QOT_OUT; i += stride)
    va.rel_impact_out[k * MI * QOT_OUT + i] = __int_as_float(0x7fc00000);
}

// the staged neighbour rows of release k, in staging order: rows with a tag (their index, < max_impact) into
// rel_impact_out, and with a bound every row's margin into r_mkey.  Lane 0.
__device__ __noinline__ void pv_rel_fold(const PvArgs& va, PvSmem& sm, const PlWarpSmem& pw, int cnt, int64_t k) {
  const PlArgs& pa = va.p;
  const int MI = pa.c.max_impact;
  for (int r = 0; r < cnt; ++r) {
    const int t = pw.rtag[r];
    if (t >= 0)
      for (int o = 0; o < QOT_OUT; ++o) va.rel_impact_out[(k * MI + t) * QOT_OUT + o] = pw.rout[r][o];
    if (pa.bound) {
      const float v = pw.rout[r][pa.metric], b = pa.bound[pw.rnode[r]];
      sm.r_mkey = min(sm.r_mkey, pl_okey(pa.maximize ? __fsub_rn(v, b) : __fsub_rn(b, v)));
    }
  }
}

// a 256-bit row with the bit at position R taken out: the bits above R move down one place
__device__ __forceinline__ void pv_remove_bit(unsigned (&r)[kCdMaskWords], int R) {
  const int wr = R >> 5, b = R & 31;
#pragma unroll
  for (int k = 0; k < kCdMaskWords; ++k) {
    const unsigned next = k + 1 < kCdMaskWords ? r[k + 1] : 0u;
    const unsigned keep = k < wr ? 0xffffffffu : k == wr ? (1u << b) - 1u : 0u;
    r[k] = (r[k] & keep) | (r[k] >> 1 & ~keep) | (k >= wr ? next << 31 : 0u);
  }
}

// the lightpath at rank sm.r_rank out of chan_work, bound_work and the block's graph: its channels -1, the highest
// stable id relabelled to its freed one, rank R removed and every row's bits above R moved down one place.  All
// threads; the caller's neighbour rows are staged before.
__device__ __noinline__ void pv_release(const PvArgs& va, PvSmem& sm, int64_t s, int64_t n0, int tid) {
  const CdArgs& a = va.p.c;
  __syncthreads();                                        // the neighbour rows are staged
  const int R = sm.r_rank, nt = sm.n_tot, last = nt - 1;
  const short sid = sm.r2s[R];
  const int LQ = a.cfg.L * a.cfg.Q;
  int32_t* row = va.chan_work + s * LQ;
  const int32_t vs = static_cast<int32_t>(n0 + sid), vl = static_cast<int32_t>(n0 + last);
  int freed = 0;
  for (int ch = tid; ch < LQ; ch += kCdThreads) {
    const int32_t v = __ldcg(row + ch);
    if (v == vs) {
      row[ch] = -1;
      ++freed;
    } else if (v == vl) {
      row[ch] = vs;
    }
  }
  if (freed) atomicSub(&sm.n_chan, freed);
  if (va.bound_work && tid == 0) va.bound_work[s * kCdMaxN + sid] = va.bound_work[s * kCdMaxN + last];
  unsigned rw[kCdMaskWords];
  float xr[kF];
  long long cn = 0;
  int ky = 0;
  short st = 0;
  const bool keep = tid < nt && tid != R;
  if (keep) {
#pragma unroll
    for (int k = 0; k < kCdMaskWords; ++k) rw[k] = sm.adj[tid][k];
    pv_remove_bit(rw, R);
#pragma unroll
    for (int k = 0; k < kF; ++k) xr[k] = sm.x[tid][k];
    cn = sm.conn[tid];
    ky = sm.key[tid];
    st = sm.r2s[tid] == last ? sid : sm.r2s[tid];
  }
  __syncthreads();
  if (keep) {
    const int to = tid < R ? tid : tid - 1;
#pragma unroll
    for (int k = 0; k < kCdMaskWords; ++k) sm.adj[to][k] = rw[k];
#pragma unroll
    for (int k = 0; k < kF; ++k) sm.x[to][k] = xr[k];
    sm.conn[to] = cn;
    sm.key[to] = ky;
    sm.r2s[to] = st;
  }
  __syncthreads();
  for (int r = tid; r < last; r += kCdThreads) sm.s2r[sm.r2s[r]] = static_cast<short>(r);
  if (tid == 0) sm.n_tot = last;
  __syncthreads();
}

// the neighbours by rank of placement [q0, q0 + cw) on route links[p0, p1), from chan_work (the route was scanned
// before: every occupied channel is free, a known node's or unknown)
__device__ __forceinline__ void pv_scan(const PvArgs& va, const PvSmem& sm, int64_t s, int64_t n0, int64_t p0,
                                        int64_t p1, int q0, int cw, unsigned* mask, int lane) {
  const CdArgs& a = va.p.c;
  for (int64_t e = p0; e < p1; ++e) {
    const int32_t* row = va.chan_work + (s * a.cfg.L + a.links[e]) * a.cfg.Q;
    for (int q = lane; q < a.cfg.Q; q += 32) {
      const int32_t v = __ldcg(row + q);
      const int64_t j = static_cast<int64_t>(v) - n0;
      if (v < 0 || j < 0 || j >= sm.n_tot || (q >= q0 && q < q0 + cw)) continue;
      if (cd_df_hit(a.freqs, a.freqs[q], q0, cw, a.cfg.freq_threshold)) {
        const int r = sm.s2r[j];
        atomicOr(&mask[r >> 5], 1u << (r & 31));
      }
    }
  }
}

// a 256-bit row with a bit inserted at position R (value v): the bits from R up move one place
__device__ __forceinline__ void pv_insert_bit(unsigned (&r)[kCdMaskWords], int R, unsigned v) {
  const int wr = R >> 5, b = R & 31;
#pragma unroll
  for (int k = kCdMaskWords - 1; k >= 0; --k) {
    const unsigned prev = k ? r[k - 1] : 0u;
    const unsigned keep = k < wr ? 0xffffffffu : k == wr ? (1u << b) - 1u : 0u;
    r[k] = (r[k] & keep) | (r[k] & ~keep) << 1 | (k > wr ? prev >> 31 : 0u) | (k == wr ? v << b : 0u);
  }
}

// the accepted demand into chan_work, bound_work and the block's graph: the new node inserted at rank R (the number of
// nodes whose first channel comes before its own), every row's bits from R up moved one place.  All threads.
__device__ __noinline__ void pv_commit(const PvArgs& va, PvSmem& sm, int64_t s, int64_t n0, int tid) {
  const PlArgs& pa = va.p;
  const CdArgs& a = pa.c;
  const int L = a.cfg.L, Q = a.cfg.Q;
  const int64_t po = sm.c_po, p0 = a.link_ptr[po], p1 = a.link_ptr[po + 1];
  const int cw = a.width[po], q0 = sm.c_q0, ck = sm.c_key, nt = sm.n_tot;
  const int64_t len = p1 - p0;
  for (int64_t k = tid; k < len * cw; k += kCdThreads)
    va.chan_work[(s * L + a.links[p0 + k / cw]) * Q + q0 + k % cw] = static_cast<int32_t>(n0 + nt);
  if (va.bound_work && tid == 0) va.bound_work[s * kCdMaxN + nt] = pa.own_bound[po];
  const int R = __syncthreads_count(tid < nt && sm.key[tid] < ck);
  unsigned rw[kCdMaskWords];
  float xr[kF];
  long long cn = 0;
  int ky = 0;
  short sid = 0;
  const bool old = tid < nt, ins = tid == kCdThreads - 1;
  if (old || ins) {
#pragma unroll
    for (int k = 0; k < kCdMaskWords; ++k) rw[k] = ins ? sm.wmask[k] : sm.adj[tid][k];
    pv_insert_bit(rw, R, ins ? 0u : sm.wmask[tid >> 5] >> (tid & 31) & 1u);
#pragma unroll
    for (int k = 0; k < kF; ++k) xr[k] = ins ? sm.cd.w[0].cx[k] : sm.x[tid][k];
    cn = ins ? sm.top + 1 : sm.conn[tid];
    ky = ins ? ck : sm.key[tid];
    sid = ins ? static_cast<short>(nt) : sm.r2s[tid];
  }
  __syncthreads();
  if (old || ins) {
    const int to = ins ? R : tid < R ? tid : tid + 1;
#pragma unroll
    for (int k = 0; k < kCdMaskWords; ++k) sm.adj[to][k] = rw[k];
#pragma unroll
    for (int k = 0; k < kF; ++k) sm.x[to][k] = xr[k];
    sm.conn[to] = cn;
    sm.key[to] = ky;
    sm.r2s[to] = sid;
  }
  __syncthreads();
  for (int r = tid; r <= nt; r += kCdThreads) sm.s2r[sm.r2s[r]] = static_cast<short>(r);
  if (tid == 0) {
    sm.n_tot = nt + 1;
    sm.n_chan += static_cast<int>(len * cw);
    sm.top += 1;
  }
  __syncthreads();
}

// Protection (qot_lightpath_protect; kProtect): a protected demand (protect[d] != 0) is placed twice against the
// block's state.  First the working path, over the options that have a link-disjoint partner among the demand's
// options (the others are skipped as restoration skips options crossing a failed link: never scanned, never counted;
// none left: QOT_PROT_NO_PARTNER).  An acceptable working path goes in with pv_commit (conn_id top + 1, its own_bound),
// then the backup path is placed the same way over the options whose route shares no link with the working route,
// its outputs written through bk (PtArgs: the backup output arrays).  An acceptable backup goes in as top + 2; else
// pv_release takes the working path out again (stable id n_tot - 1, the highest: nothing is relabelled) and top goes
// back, so the state is what it was before the demand.  The link sets are 1024-bit bitmaps (QOT_TG_MAX_LINKS), word
// t held in bm[t].  An unprotected demand is handled exactly as without kProtect, its backup outputs empty.
struct PtSmem {
  PvSmem v;                                  // lp_provision_kernel's block state
  unsigned bm[QOT_TG_MAX_LINKS / 32];        // a route's links
  unsigned skip;                             // the current search's options skipped (bit po - o0)
};
static_assert(sizeof(PtSmem) + 16 <= 227 * 1024, "lp_provision_kernel<.., true>: shared memory over the 227 KB limit");
static_assert(QOT_TG_MAX_LINKS == 32 * 32 && kPlMaxOptions <= 32, "one bitmap word per lane, one skip bit per option");

struct PtArgs : PvArgs {
  PvArgs bk;                               // the same arguments with the backup output arrays
  const uint8_t* protect;                  // [D] or null (none protected)
};
template <bool kProtect>
using PvKernelArgs = std::conditional_t<kProtect, PtArgs, PvArgs>;

// route links[p0, p1) into the bitmap bm (all lanes of one warp; links checked to lie in [0, QOT_TG_MAX_LINKS))
__device__ __forceinline__ void pt_route_bits(const CdArgs& a, int64_t p0, int64_t p1, unsigned* bm, int lane) {
  bm[lane] = 0u;
  __syncwarp();
  for (int64_t e = p0 + lane; e < p1; e += 32) atomicOr(&bm[a.links[e] >> 5], 1u << (a.links[e] & 31));
  __syncwarp();
}

// true on every lane when route links[p0, p1) shares a link with bm
__device__ __forceinline__ bool pt_touches(const CdArgs& a, int64_t p0, int64_t p1, const unsigned* bm, int lane) {
  bool hit = false;
  for (int64_t e = p0 + lane; e < p1 && !hit; e += 32) hit = bm[a.links[e] >> 5] >> (a.links[e] & 31) & 1u;
  return __any_sync(kFull, hit);
}

// the arguments a search writes its outputs through: the backup's in the backup search (ph = 1), else the demand's
template <bool kProtect>
__device__ __forceinline__ const PvArgs& pv_out_args(const PvKernelArgs<kProtect>& args, int ph) {
  if constexpr (kProtect) return ph ? static_cast<const PvArgs&>(args.bk) : static_cast<const PvArgs&>(args);
  else return args;
}

template <bool kReleases, bool kProtect = false>
__global__ void __launch_bounds__(kCdThreads, 1) lp_provision_kernel(const __grid_constant__ PvKernelArgs<kProtect> args) {
  const PvArgs& va = args;
  const PlArgs& pa = va.p;
  const CdArgs& a = pa.c;
  PvSmem& sm = *reinterpret_cast<PvSmem*>(cd_smem_raw);
  PtSmem& pt = *reinterpret_cast<PtSmem*>(cd_smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = sm.cd.w[w];
  PlWarpSmem& pw = sm.w[w];
  float As[kF], Ad[kF];
  cd_head_prologue(a.prep, As, Ad, tid);
  if (tid == 0) sm.n_valid = sm.n_rvalid = 0ull;
  // ---- the grouping, checked whole by every block: sample_ptr non-decreasing from 0; order[i] a demand of the sample
  // whose range holds i, ascending within the range; the ranges hold every demand with a sample in [0, S).  The same
  // for the releases, ordered by (before, k) within a range.  Otherwise no demand is provisioned and no release
  // applied: every output says PROV_BAD_GROUPING, each written by exactly one thread of the grid.
  const int64_t S = a.S, D = a.K, NR = kReleases ? va.rel.R : 0;
  bool bad = false;
  for (int64_t g = tid; g <= S; g += kCdThreads) {
    const int64_t v = va.sample_ptr[g];
    bad |= (g == 0 && v != 0) || (g < S && va.sample_ptr[g + 1] < v) || (g == S && v > D);
  }
  bad = __syncthreads_or(bad);
  if (!bad) {
    const int64_t nv = va.sample_ptr[S];
    unsigned long long cnt = 0;
    for (int64_t i = tid; i < D; i += kCdThreads) {
      const int64_t sd = a.sample[i];
      cnt += sd >= 0 && sd < S;
      if (i < nv) {
        const int64_t d = va.order[i];
        bool ok = d >= 0 && d < D;
        const int64_t s = ok ? a.sample[d] : -1;
        ok = ok && s >= 0 && s < S && va.sample_ptr[s] <= i && i < va.sample_ptr[s + 1];
        if (ok && i + 1 < va.sample_ptr[s + 1]) ok = va.order[i + 1] > d;
        bad |= !ok;
      }
    }
    atomicAdd(&sm.n_valid, cnt);
    bad = __syncthreads_or(bad) || sm.n_valid != static_cast<unsigned long long>(nv);
  }
  if (!bad && NR > 0) {
    const int64_t* rp = va.rel_ptr;
    const int64_t* bf = va.rel.before;
    for (int64_t g = tid; g <= S; g += kCdThreads) {
      const int64_t v = rp[g];
      bad |= (g == 0 && v != 0) || (g < S && rp[g + 1] < v) || (g == S && v > NR);
    }
    bad = __syncthreads_or(bad);
    if (!bad) {
      const int64_t nv = rp[S];
      unsigned long long cnt = 0;
      for (int64_t i = tid; i < NR; i += kCdThreads) {
        const int64_t sk = va.rel.sample[i];
        cnt += sk >= 0 && sk < S;
        if (i < nv) {
          const int64_t k = va.rel_order[i];
          bool ok = k >= 0 && k < NR;
          const int64_t s = ok ? va.rel.sample[k] : -1;
          ok = ok && s >= 0 && s < S && rp[s] <= i && i < rp[s + 1];
          if (ok && i + 1 < rp[s + 1]) {
            const int64_t k2 = va.rel_order[i + 1];
            ok = k2 >= 0 && k2 < NR && (bf[k2] > bf[k] || (bf[k2] == bf[k] && k2 > k));
          }
          bad |= !ok;
        }
      }
      atomicAdd(&sm.n_rvalid, cnt);
      bad = __syncthreads_or(bad) || sm.n_rvalid != static_cast<unsigned long long>(nv);
    }
  }
  const int64_t gt = static_cast<int64_t>(blockIdx.x) * kCdThreads + tid;
  const int64_t gs = static_cast<int64_t>(gridDim.x) * kCdThreads;
  if (bad) {
    for (int64_t d = gt; d < D; d += gs) pv_empty(va, d, QOT_PROV_BAD_GROUPING, 0, 1);
    for (int64_t k = gt; k < NR; k += gs) pv_rel_empty(va, k, QOT_PROV_BAD_GROUPING, 0, 0, 1);
    if constexpr (kProtect)
      for (int64_t d = gt; d < D; d += gs) pv_empty(args.bk, d, 0, 0, 1);
    return;
  }
  for (int64_t d = gt; d < D; d += gs)
    if (a.sample[d] < 0 || a.sample[d] >= S) pv_empty(va, d, QOT_CAND_BAD_SAMPLE, 0, 1);
  if constexpr (kProtect)
    for (int64_t d = gt; d < D; d += gs)
      if (a.sample[d] < 0 || a.sample[d] >= S) pv_empty(args.bk, d, 0, 0, 1);
  for (int64_t k = gt; k < NR; k += gs)
    if (va.rel.sample[k] < 0 || va.rel.sample[k] >= S) pv_rel_empty(va, k, QOT_CAND_BAD_SAMPLE, 0, 0, 1);
  const float nan = __int_as_float(0x7fc00000);
  int zc = 0;                                             // rows staged in this warp's head buffer
  for (int64_t s = blockIdx.x; s < S; s += gridDim.x) {
    const int64_t i0 = va.sample_ptr[s], i1 = va.sample_ptr[s + 1];
    const int64_t j0 = NR > 0 ? va.rel_ptr[s] : 0, j1 = NR > 0 ? va.rel_ptr[s + 1] : 0;
    if (i0 == i1 && j0 == j1) continue;
    const int L = a.cfg.L, Q = a.cfg.Q;
    int64_t n0 = 0;
    int n = 0;
    const bool state_ok = cd_sample_nodes(a, s, n0, n);
    // ---- the sample's graph, in node order: adjacency from the out-runs, x, conn_ids, first channels, bounds
    __syncthreads();                                      // the previous sample's graph is no longer read
    for (int i = tid; i < kCdMaxN * kCdMaskWords; i += kCdThreads) (&sm.adj[0][0])[i] = 0u;
    for (int r = tid; r < kCdMaxN; r += kCdThreads) {
      sm.key[r] = INT_MAX;
      sm.r2s[r] = sm.s2r[r] = static_cast<short>(r);
    }
    if (tid == 0) {
      sm.n_tot = state_ok ? n : 0;
      sm.n_chan = 0;
      sm.top = 0;
    }
    __syncthreads();
    bool sbad = !state_ok;
    if (state_ok) {
      for (int r = w; r < n; r += kCdWarps) sbad |= !cd_old_nbrs(a, n0, n, r, sm.adj[r], lane);
      for (int i = tid; i < n * kF; i += kCdThreads) (&sm.x[0][0])[i] = a.x[n0 * kF + i];
      long long top = 0;
      for (int r = tid; r < n; r += kCdThreads) {
        const long long c = va.conn_ids[n0 + r];
        sm.conn[r] = c;
        top = max(top, c);
      }
      atomicMax(&sm.top, top);
      int nch = 0;
      const int32_t* crow = va.chan_work + s * L * Q;
      for (int ch = tid; ch < L * Q; ch += kCdThreads) {
        const int32_t v = __ldcg(crow + ch);
        if (v == -1) continue;
        ++nch;
        const int64_t j = static_cast<int64_t>(v) - n0;
        if (v >= 0 && j >= 0 && j < n) atomicMin(&sm.key[j], ch);
      }
      atomicAdd(&sm.n_chan, nch);
      if (va.bound_work)
        for (int r = tid; r < n; r += kCdThreads) va.bound_work[s * kCdMaxN + r] = va.bound[n0 + r];
    }
    sbad = __syncthreads_or(sbad);
    int64_t j = j0;                                       // the sample's next release
    for (int64_t i = i0; i <= i1; ++i) {
      const int64_t d = i < i1 ? va.order[i] : -1;
      // ---- the releases due before demand d (after the last demand: the rest)
      for (; j < j1 && (i == i1 || va.rel.before[va.rel_order[j]] <= d); ++j) {
        const int64_t k = va.rel_order[j];
        if (tid == 0) {                                   // what it names: status and conn_id
          const int64_t b = va.rel.before[k], dm = va.rel.demand[k];
          int rs = 0;
          long long c = -1;
          if (sbad) rs = QOT_CAND_BAD_STATE;
          else if (b < 0 || b > D || dm < -1 || (dm >= 0 && (dm >= D || dm >= b || a.sample[dm] != s)))
            rs = QOT_TRAF_BAD_REF;
          else if (dm >= 0 && (c = __ldcg(va.conn_id + dm)) < 0) rs = QOT_TRAF_NOT_ACCEPTED;
          else if (dm == -1) c = va.rel.conn_id[k];
          sm.r_st = rs;
          sm.r_conn = c;
          sm.r_rank = -1;
          sm.r_mkey = 0xffffffffu;
        }
        __syncthreads();
        if (sm.r_st == 0 && tid < sm.n_tot && sm.conn[tid] == sm.r_conn) sm.r_rank = tid;
        __syncthreads();
        const int R = sm.r_rank;
        // ---- warp 0: the former neighbours' rows (all of them against a bound) and the release's outputs
        if (w == 0) {
          if (zc) {                                       // the previous demand's winner rows
            pl_flush(pa, pw, w, zc, 0, lane);
            zc = 0;
          }
          const int rs = sm.r_st ? sm.r_st : R < 0 ? QOT_TRAF_BAD_REF : 0;
          if (rs) {
            pv_rel_empty(va, k, rs, 0, lane, 32);
          } else {
            const int MI = a.max_impact;
            const int cnt = cd_rank(lane < kCdMaskWords ? sm.adj[R][lane] : 0u, ws.nbr, lane);
            __syncwarp();
            const int rows = min(cnt, MI), nev = pa.bound ? cnt : rows;
            const auto flush = [&](int c) {
              cd_flush(w, c, a.prep, lane);
              if (lane == 0) pv_rel_fold(va, sm, pw, c, k);
              __syncwarp();
            };
            for (int e = 0; e < nev; ++e) {
              const int r = ws.nbr[e];
              if (lane == 0 && e < rows) va.rel_impact_conn[k * MI + e] = sm.conn[r];
              const unsigned rb = lane == R >> 5 ? 1u << (R & 31) : 0u;
              const int m = cd_rank(lane < kCdMaskWords ? sm.adj[r][lane] & ~rb : 0u, ws.msg, lane);
              if (lane == 0) {
                ws.msg[m] = r;
                pw.rtag[zc] = e < rows ? e : -1;
                pw.rnode[zc] = s * kCdMaxN + sm.r2s[r];
              }
              __syncwarp();
              zc = cd_row(ws, zc, ws.msg, m + 1, r, PvX{sm.x, ws.cx, r, a.lut_col}, As, Ad, pw.rout[zc], flush, lane);
            }
            if (zc) {
              flush(zc);
              zc = 0;
            }
            pv_rel_empty(va, k, 0, rows, lane, 32);
            if (lane == 0) {
              va.rel_status[k] = cnt > MI ? QOT_CAND_IMPACT_OVERFLOW : 0;
              va.rel_conn_id[k] = sm.r_conn;
              va.rel_n_impact[k] = cnt;
              va.rel_margin[k] = pa.bound && cnt ? pl_unkey(sm.r_mkey) : nan;
            }
          }
        }
        if (R >= 0) pv_release(va, sm, s, n0, tid);
        __syncthreads();                                  // the release's shared state is read
      }
      if (i == i1) break;
      const int64_t o0 = pa.opt_ptr[d], o1 = pa.opt_ptr[d + 1];
      [[maybe_unused]] bool prot = false;                 // kProtect: d is protected
      [[maybe_unused]] int ph = 0;                        // kProtect: 0 the working path, 1 the backup
      if constexpr (kProtect) prot = args.protect && args.protect[d];
    search:                                               // kProtect: the backup search starts here again
      // ---- validation (warp 0): the option range, every option's route and width; then the state
      if (w == 0) {
        const bool opts_ok = o0 >= 0 && o1 > o0 && o1 <= pa.P && o1 - o0 <= kPlMaxOptions;
        bool badp = !opts_ok;
        if (opts_ok)
          for (int64_t po = o0; po < o1 && !badp; ++po) {
            const int cw = a.width[po];
            badp = cd_bad_route(a, L, a.link_ptr[po], a.link_ptr[po + 1], false, cw < 1 || cw > Q, lane);
          }
        if (lane == 0) sm.st = badp ? QOT_CAND_BAD_PATH : sbad ? QOT_CAND_BAD_STATE : 0;
        if constexpr (kProtect) {
          // working: the options without a link-disjoint partner; backup: those sharing a link with the working route
          unsigned skip = 0u;
          if (prot && !badp) {
            if (ph == 0) {
              for (int64_t po = o0; po < o1; ++po) {
                pt_route_bits(a, a.link_ptr[po], a.link_ptr[po + 1], pt.bm, lane);
                bool partner = false;
                for (int64_t p2 = o0; p2 < o1 && !partner; ++p2)
                  partner = !pt_touches(a, a.link_ptr[p2], a.link_ptr[p2 + 1], pt.bm, lane);
                if (!partner) skip |= 1u << (po - o0);
              }
            } else {                                      // sm.c_po: the working option, committed
              pt_route_bits(a, a.link_ptr[sm.c_po], a.link_ptr[sm.c_po + 1], pt.bm, lane);
              for (int64_t po = o0; po < o1; ++po)
                if (pt_touches(a, a.link_ptr[po], a.link_ptr[po + 1], pt.bm, lane)) skip |= 1u << (po - o0);
            }
          }
          if (lane == 0) {
            pt.skip = skip;
            if (prot && !badp && !sbad && skip == (o1 - o0 >= 32 ? 0xffffffffu : (1u << (o1 - o0)) - 1u))
              sm.st = QOT_PROT_NO_PARTNER;
          }
        }
      }
      if (lane == 0) {
        pw.key = 0ull;
        pw.n_free = pw.n_feas = 0;
      }
      __syncthreads();
      const auto row = [&](const int* msg, int M, int q, float* dst, int tag, long long node) {
        if (lane == 0) {
          pw.rtag[zc] = tag;
          pw.rnode[zc] = node;
        }
        zc = cd_row(ws, zc, msg, M, q, PvX{sm.x, ws.cx, q, a.lut_col}, As, Ad, dst ? dst : pw.rout[zc],
                    [&](int cnt) { pl_flush(pa, pw, w, cnt, o0, lane); }, lane);
      };
      int st = sm.st;                                     // block-uniform
      int seq = 0, wseq = 0;                              // placements of this demand: all, this warp's
      [[maybe_unused]] unsigned skip = 0u;
      if constexpr (kProtect) skip = pt.skip;
      for (int64_t po = o0; st == 0 && po < o1; ++po) {
        if constexpr (kProtect)
          if (skip >> (po - o0) & 1u) continue;
        const int64_t p0 = a.link_ptr[po], p1 = a.link_ptr[po + 1];
        const int cw = a.width[po];
        // ---- warp 0: the route's occupied bitmap and its channels of known lightpaths by rank, one read per row
        if (w == 0) {
          unsigned occ = 0u;
          int ne = 0;
          bool rbad = false;
          const int nt = sm.n_tot;
          for (int64_t e = p0; e < p1; ++e) {
            const int32_t* crow = va.chan_work + (s * L + a.links[e]) * Q;
            for (int qb = 0; qb < Q; qb += 32) {
              const int q = qb + lane;
              const int32_t v = q < Q ? __ldcg(crow + q) : -1;
              const unsigned ob = __ballot_sync(kFull, v != -1);
              if (lane == qb >> 5) occ |= ob;
              const int64_t j = static_cast<int64_t>(v) - n0;
              const bool known = v >= 0 && j >= 0 && j < nt;
              rbad |= v >= 0 && !known;
              const unsigned kb = __ballot_sync(kFull, known);
              const int at = ne + __popc(kb & ((1u << lane) - 1u));
              if (known && at < kPlEntCap) sm.ent[at] = q << 8 | sm.s2r[j];
              ne += __popc(kb);
            }
          }
          sm.run[lane] = pl_free_starts(occ, Q, cw, lane);
          rbad = __any_sync(kFull, rbad);
          if (lane == 0) {
            sm.ne = ne;
            sm.rbad = rbad;
          }
        }
        __syncthreads();
        if (sm.rbad) {
          st |= QOT_CAND_BAD_STATE;
          break;
        }
        // ---- the free starts in ascending order, dealt round-robin to the warps
        const int ne = sm.ne;
        for (int wd = 0; wd < 32 && 32 * wd < Q; ++wd) {
          for (unsigned bits = sm.run[wd]; bits; bits &= bits - 1u) {
            const int q0 = 32 * wd + __ffs(bits) - 1;
            if (seq++ % kCdWarps != w) continue;
            if (lane < kCdMaskWords) ws.mask[lane] = 0u;
            __syncwarp();
            if (ne <= kPlEntCap) pl_ent_mask(a, sm.ent, ne, q0, cw, ws.mask, lane);
            else pv_scan(va, sm, s, n0, p0, p1, q0, cw, ws.mask, lane);
            __syncwarp();
            const int nn = cd_rank(lane < kCdMaskWords ? ws.mask[lane] : 0u, ws.nbr, lane);
            cd_xrow(a, ws.cx, [&] { return lane == 0 ? static_cast<float>(a.freqs[q0]) : a.feat[po * 3 + lane - 1]; },
                    lane);
            const int slot = wseq++ & (kPlRing - 1);
            const int nimp = pa.bound ? nn : 0;           // impact rows count against a bound, all of them
            if (lane == 0) {
              ws.nbr[nn] = kCand;
              PlPending& pp = pw.ring[slot];
              pp.mkey = 0xffffffffu;
              pp.left = 1 + nimp;
              pp.p = static_cast<int>(po);
              pp.q0 = q0;
              ++pw.n_free;
            }
            __syncwarp();
            row(ws.nbr, nn + 1, kCand, nullptr, slot, -1);
            for (int k = 0; k < nimp; ++k) {
              const int r = ws.nbr[k];
              const int m = cd_rank(lane < kCdMaskWords ? sm.adj[r][lane] : 0u, ws.msg, lane);
              if (lane == 0) {
                ws.msg[m] = kCand;
                ws.msg[m + 1] = r;
              }
              __syncwarp();
              row(ws.msg, m + 2, r, nullptr, slot, s * kCdMaxN + sm.r2s[r]);
            }
          }
        }
        __syncthreads();                                  // the entries and free words are read
      }
      // ---- every placement folded: the block's winner and counts
      if (zc) {
        pl_flush(pa, pw, w, zc, o0, lane);
        zc = 0;
      }
      __syncthreads();
      if (tid == 0) {
        unsigned long long key = 0ull;
        int nf = 0, nfe = 0, bw = -1;
        for (int v = 0; v < kCdWarps; ++v) {
          nf += sm.w[v].n_free;
          nfe += sm.w[v].n_feas;
          if (sm.w[v].key > key) {
            key = sm.w[v].key;
            bw = v;
          }
        }
        sm.key_best = key;
        sm.n_free = nf;
        sm.n_feas = nfe;
        if (bw >= 0)
          for (int o = 0; o < 4; ++o) sm.best[o] = sm.w[bw].best[o];
      }
      __syncthreads();
      // ---- warp 0: the winner's impact rows and the demand's outputs; acceptance
      if (w == 0) {
        // the outputs written: the demand's, or with kProtect in the backup search the backup's
        const PvArgs& vo = pv_out_args<kProtect>(args, ph);
        const PlArgs& po_ = vo.p;
        const CdArgs& ao = po_.c;
        const int MI = a.max_impact;
        const unsigned long long key = sm.key_best;
        int cnt = 0, rows = 0, bp = -1, bq = -1;
        int64_t po = -1, p0 = 0, p1 = 0;
        int cw = 0;
        if (st == 0 && key) {
          const unsigned idx = 0xffffffffu - static_cast<unsigned>(key);
          bp = static_cast<int>(idx >> 10);
          bq = static_cast<int>(idx & 1023u);
          po = o0 + bp;
          p0 = a.link_ptr[po];
          p1 = a.link_ptr[po + 1];
          cw = a.width[po];
          if (lane < kCdMaskWords) sm.wmask[lane] = 0u;
          __syncwarp();
          pv_scan(va, sm, s, n0, p0, p1, bq, cw, sm.wmask, lane);
          __syncwarp();
          cnt = cd_rank(lane < kCdMaskWords ? sm.wmask[lane] : 0u, ws.nbr, lane);
          rows = min(cnt, MI);
          cd_xrow(a, ws.cx, [&] { return lane == 0 ? static_cast<float>(a.freqs[bq]) : a.feat[po * 3 + lane - 1]; },
                  lane);
          __syncwarp();
          for (int k = 0; k < rows; ++k) {
            const int r = ws.nbr[k];
            if (lane == 0) ao.impact_node[d * MI + k] = sm.conn[r];
            const int m = cd_rank(lane < kCdMaskWords ? sm.adj[r][lane] : 0u, ws.msg, lane);
            if (lane == 0) {
              ws.msg[m] = kCand;
              ws.msg[m + 1] = r;
            }
            __syncwarp();
            row(ws.msg, m + 2, r, ao.impact_out + (d * MI + k) * QOT_OUT, -1, -1);
          }
        }
        if (st & (kProtect ? kPlFatal | QOT_PROT_NO_PARTNER : kPlFatal)) {
          pv_empty(vo, d, st, lane, 32);
          if (lane == 0) sm.acc = 0;
        } else {
          cd_clear_impact(ao, d, rows, MI, nullptr, lane, 32);
          // the graph builder refuses a sample over QOT_TG_MAX_NODES lightpaths or QOT_TG_MAX_CHANNELS channels
          const bool full = key && (sm.n_tot >= kCdMaxN || sm.n_chan + (p1 - p0) * cw > QOT_TG_MAX_CHANNELS);
          const bool acc = key && !full;
          int first = INT_MAX;                            // the accepted lightpath's first channel
          for (int64_t e = p0 + lane; acc && e < p1; e += 32) first = min(first, a.links[e] * Q + bq);
          first = __reduce_min_sync(kFull, first);
          if (lane < QOT_OUT) ao.out[d * QOT_OUT + lane] = key ? sm.best[lane] : nan;
          if (lane == 0) {
            ao.status[d] = st | (cnt > MI ? QOT_CAND_IMPACT_OVERFLOW : 0) | (full ? QOT_PROV_FULL : 0);
            ao.n_impact[d] = cnt;
            po_.option[d] = bp;
            po_.q0[d] = bq;
            po_.margin[d] = key ? sm.best[3] : nan;
            po_.n_free[d] = sm.n_free;
            po_.n_feasible[d] = sm.n_feas;
            vo.conn_id[d] = acc ? sm.top + 1 : -1;
            sm.acc = acc;
            sm.c_po = po;
            sm.c_q0 = bq;
            sm.c_key = first;
          }
        }
        if constexpr (kProtect) {
          __syncwarp();
          const bool acc = sm.acc;
          if (ph == 0 && !(prot && acc)) pv_empty(args.bk, d, 0, lane, 32);   // no backup search: empty
          if (ph == 1 && !acc && lane == 0) {             // no backup: the demand is not accepted
            a.status[d] |= QOT_PROT_NO_BACKUP;
            va.conn_id[d] = -1;
          }
        }
      }
      __syncthreads();
      if constexpr (kProtect) {
        if (ph == 1 && !sm.acc) {                         // the working path out again, top back
          if (tid == 0) {
            sm.r_rank = sm.s2r[sm.n_tot - 1];
            sm.top -= 1;
          }
          pv_release(va, sm, s, n0, tid);
          continue;
        }
      }
      if (!sm.acc) continue;
      pv_commit(va, sm, s, n0, tid);
      if (kProtect && prot && ph == 0) {                  // the working path is in: its backup
        ph = 1;
        goto search;
      }
    }
  }
  if (zc) pl_flush(pa, pw, w, zc, 0, lane);
}

// ------------------------------------------------------------------------------------------------ restoration
// lp_restore_kernel: persistent, one block per failure scenario (qot_lightpath_restore).  Scenario f names a sample s
// and a set of failed links; any number of scenarios may name one sample, so the block works on its own slabs,
// chan_work[b] and bound_work[b] (b = blockIdx.x), never on a slab of the sample's.  Per scenario:
//   s's chan_node row is copied into chan_work[b], bound into bound_work[b] and the dense graph loaded as
//     lp_provision_kernel loads it (rank = node order);
//   the failed links' chan_node rows give the cut set C, a 256-bit mask by sample-local node; pv_release takes each
//     cut lightpath out, highest node first (a release relabels only the highest stable id, so a lower node's stable
//     id is still its node index when its turn comes), without its neighbours' rows;
//   each c in C, ascending, is a demand with c's options (options.opt_ptr[n0 + c]), placed as lp_provision_kernel
//     places a demand; an option whose route touches a failed link is skipped (bit po - o0 of `skip`): never scanned,
//     never counted.  Option indices stay those of c's full list, so the tie rule (the lower index wins) is that of
//     the filtered list.  An accepted demand goes in with pv_commit, then takes c's conn_id back;
//   every remaining rank's row (its adjacency row by rank, then its self loop: the every-node row of the end state)
//     goes through the same head, 12 warps round-robin, folded into end_margin / n_below and written to end_out.
// The demand body is lp_provision_kernel's without the impact rows, so a restoration's outputs are bit-identical to
// qot_lightpath_traffic's for the same releases and filtered demands.
struct RsSmem {
  PvSmem v;                                  // lp_provision_kernel's block state (head, warps, dense graph)
  unsigned cut[kCdMaskWords];                // the cut set by sample-local node
  unsigned skip;                             // the current demand's options that touch a failed link
  unsigned e_mkey;                           // min of the end rows' margin keys
  int e_below, f_st, n_rest;
  long long c_conn;                          // the current demand's conn_id
};
static_assert(sizeof(RsSmem) + 16 <= 227 * 1024, "lp_restore_kernel: shared memory over the 227 KB block limit");

struct RsArgs {
  PvArgs v;                                // v.p.c.chan_node = v.chan_work = the [blocks, L, Q] slabs, v.p.bound =
                                           // v.bound_work (or null); demand outputs at f * max_cut + i
  const int32_t* chan_node;                // the state's [S, L, Q]
  qot_lp_failures_t fail;
  int max_cut;
  int64_t* cut_node;                       // [F, max_cut]
  int32_t* status;                         // [F]
  int32_t* n_cut;
  int32_t* n_restored;
  float* end_margin;
  int32_t* n_below;
  int64_t* end_conn;                       // [F, kCdMaxN] or null
  float* end_out;                          // [F, kCdMaxN, 3] or null
};

// the staged end rows, in staging order: their outputs into end_out (rtag: the rank) and, with a bound, their margins
// into e_mkey / e_below.  Lane 0.
__device__ __noinline__ void rs_end_fold(const RsArgs& ra, RsSmem& rs, const PlWarpSmem& pw, int cnt, int64_t f) {
  const PlArgs& pa = ra.v.p;
  for (int r = 0; r < cnt; ++r) {
    if (ra.end_out)
      for (int o = 0; o < QOT_OUT; ++o) ra.end_out[(f * kCdMaxN + pw.rtag[r]) * QOT_OUT + o] = pw.rout[r][o];
    if (pa.bound) {
      const float v = pw.rout[r][pa.metric], b = pa.bound[pw.rnode[r]];
      const unsigned k = pl_okey(pa.maximize ? __fsub_rn(v, b) : __fsub_rn(b, v));
      atomicMin(&rs.e_mkey, k);
      if (k < 0x80000000u) atomicAdd(&rs.e_below, 1);    // margin < 0 or NaN
    }
  }
}

__global__ void __launch_bounds__(kCdThreads, 1) lp_restore_kernel(const __grid_constant__ RsArgs ra) {
  const PvArgs& va = ra.v;
  const PlArgs& pa = va.p;
  const CdArgs& a = pa.c;
  RsSmem& rs = *reinterpret_cast<RsSmem*>(cd_smem_raw);
  PvSmem& sm = rs.v;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = sm.cd.w[w];
  PlWarpSmem& pw = sm.w[w];
  float As[kF], Ad[kF];
  cd_head_prologue(a.prep, As, Ad, tid);
  const float nan = __int_as_float(0x7fc00000);
  const int64_t b = blockIdx.x;                           // the block's slabs
  const int MC = ra.max_cut;
  int zc = 0;                                             // rows staged in this warp's head buffer
  for (int64_t f = blockIdx.x; f < ra.fail.F; f += gridDim.x) {
    const int L = a.cfg.L, Q = a.cfg.Q;
    // ---- the scenario: its sample, its failed links, the sample's offsets
    const int64_t s = ra.fail.sample[f];
    const int64_t l0 = ra.fail.link_ptr[f], l1 = ra.fail.link_ptr[f + 1];
    int fst = s < 0 || s >= a.S ? QOT_CAND_BAD_SAMPLE
              : !(l0 >= 0 && l1 > l0 && l1 <= ra.fail.n_links) ? QOT_REST_BAD_FAILURE : 0;
    bool lbad = false;
    for (int64_t e = l0 + tid; fst == 0 && e < l1; e += kCdThreads) lbad |= ra.fail.links[e] < 0 || ra.fail.links[e] >= L;
    int64_t n0 = 0;
    int n = 0;
    if (__syncthreads_or(lbad)) fst = QOT_REST_BAD_FAILURE;   // also: the previous scenario's state is no longer read
    if (fst == 0 && !cd_sample_nodes(a, s, n0, n)) fst = QOT_CAND_BAD_STATE;
    // ---- the sample's graph, in node order, and the block's slabs
    for (int i = tid; i < kCdMaxN * kCdMaskWords; i += kCdThreads) (&sm.adj[0][0])[i] = 0u;
    for (int r = tid; r < kCdMaxN; r += kCdThreads) {
      sm.key[r] = INT_MAX;
      sm.r2s[r] = sm.s2r[r] = static_cast<short>(r);
    }
    if (tid < kCdMaskWords) rs.cut[tid] = 0u;
    if (tid == 0) {
      sm.n_tot = fst == 0 ? n : 0;
      sm.n_chan = 0;
      sm.top = 0;
      rs.e_mkey = 0xffffffffu;
      rs.e_below = rs.n_rest = 0;
    }
    __syncthreads();
    bool sbad = false;
    if (fst == 0) {
      for (int r = w; r < n; r += kCdWarps) sbad |= !cd_old_nbrs(a, n0, n, r, sm.adj[r], lane);
      for (int i = tid; i < n * kF; i += kCdThreads) (&sm.x[0][0])[i] = a.x[n0 * kF + i];
      for (int r = tid; r < n; r += kCdThreads) sm.conn[r] = va.conn_ids[n0 + r];
      int nch = 0;
      const int32_t* crow = ra.chan_node + s * L * Q;
      int32_t* wrow = va.chan_work + b * L * Q;
      for (int ch = tid; ch < L * Q; ch += kCdThreads) {
        const int32_t v = crow[ch];
        wrow[ch] = v;
        if (v == -1) continue;
        ++nch;
        const int64_t j = static_cast<int64_t>(v) - n0;
        if (v >= 0 && j >= 0 && j < n) atomicMin(&sm.key[j], ch);
      }
      atomicAdd(&sm.n_chan, nch);
      if (va.bound_work)
        for (int r = tid; r < n; r += kCdThreads) va.bound_work[b * kCdMaxN + r] = va.bound[n0 + r];
      // the cut set: every known lightpath with a channel on a failed link
      for (int64_t e = l0; e < l1; ++e) {
        const int32_t* frow = crow + static_cast<int64_t>(ra.fail.links[e]) * Q;
        for (int q = tid; q < Q; q += kCdThreads) {
          const int64_t j = static_cast<int64_t>(frow[q]) - n0;
          if (frow[q] >= 0 && j >= 0 && j < n) atomicOr(&rs.cut[j >> 5], 1u << (j & 31));
        }
      }
    }
    if (__syncthreads_or(sbad)) fst = QOT_CAND_BAD_STATE;
    if (fst) {
      if (tid < kCdMaskWords) rs.cut[tid] = 0u;
      if (tid == 0) sm.n_tot = 0;
      __syncthreads();
    }
    // ---- the cut lightpaths out, highest node first
    int ncut = 0;
#pragma unroll 1
    for (int wd = kCdMaskWords - 1; wd >= 0; --wd)
      for (unsigned bits = rs.cut[wd]; bits; ++ncut) {
        const int hb = 31 - __clz(bits);
        bits &= ~(1u << hb);
        if (tid == 0) sm.r_rank = sm.s2r[32 * wd + hb];
        pv_release(va, sm, b, n0, tid);
      }
    // ---- each cut lightpath, ascending, placed on its options that avoid the failed links
    int i = 0;                                            // the cut lightpath's ordinal
#pragma unroll 1
    for (int wd = 0; wd < kCdMaskWords; ++wd)
      for (unsigned bits = rs.cut[wd]; bits; bits &= bits - 1u, ++i) {
        const int c = 32 * wd + __ffs(bits) - 1;
        const int64_t v = n0 + c, k = f * MC + i;         // k: the output row (i < max_cut)
        const int64_t o0 = pa.opt_ptr[v], o1 = pa.opt_ptr[v + 1];
        // ---- validation (warp 0): the sample, the option range, every option's route and width; the skip mask
        if (w == 0) {
          const bool opts_ok = o0 >= 0 && o1 >= o0 && o1 <= pa.P && o1 - o0 <= kPlMaxOptions;
          bool badp = !opts_ok;
          unsigned skip = 0u;
          for (int64_t po = o0; opts_ok && po < o1 && !badp; ++po) {
            const int cw = a.width[po];
            const int64_t p0 = a.link_ptr[po], p1 = a.link_ptr[po + 1];
            badp = cd_bad_route(a, L, p0, p1, false, cw < 1 || cw > Q, lane);
            bool hit = false;
            for (int64_t e = p0 + lane; !badp && e < p1; e += 32)
              for (int64_t g = l0; g < l1 && !hit; ++g) hit = a.links[e] == ra.fail.links[g];
            if (__any_sync(kFull, hit)) skip |= 1u << (po - o0);
          }
          if (lane == 0) {
            const unsigned all = o1 - o0 >= 32 ? 0xffffffffu : (1u << (o1 - o0)) - 1u;
            sm.st = a.sample[v] != s ? QOT_CAND_BAD_SAMPLE : badp ? QOT_CAND_BAD_PATH
                    : skip == all ? QOT_REST_NO_OPTION : 0;
            rs.skip = skip;
            rs.c_conn = va.conn_ids[v];
          }
        }
        if (lane == 0) {
          pw.key = 0ull;
          pw.n_free = pw.n_feas = 0;
        }
        __syncthreads();
        const auto row = [&](const int* msg, int M, int q, float* dst, int tag, long long node) {
          if (lane == 0) {
            pw.rtag[zc] = tag;
            pw.rnode[zc] = node;
          }
          zc = cd_row(ws, zc, msg, M, q, PvX{sm.x, ws.cx, q, a.lut_col}, As, Ad, dst ? dst : pw.rout[zc],
                      [&](int cnt) { pl_flush(pa, pw, w, cnt, o0, lane); }, lane);
        };
        int st = sm.st;                                   // block-uniform
        const unsigned skip = rs.skip;
        int seq = 0, wseq = 0;                            // placements of this demand: all, this warp's
        for (int64_t po = o0; st == 0 && po < o1; ++po) {
          if (skip >> (po - o0) & 1u) continue;
          const int64_t p0 = a.link_ptr[po], p1 = a.link_ptr[po + 1];
          const int cw = a.width[po];
          // ---- warp 0: the route's occupied bitmap and its channels of known lightpaths by rank, one read per row
          if (w == 0) {
            unsigned occ = 0u;
            int ne = 0;
            bool rbad = false;
            const int nt = sm.n_tot;
            for (int64_t e = p0; e < p1; ++e) {
              const int32_t* crow = va.chan_work + (b * L + a.links[e]) * Q;
              for (int qb = 0; qb < Q; qb += 32) {
                const int q = qb + lane;
                const int32_t cv = q < Q ? __ldcg(crow + q) : -1;
                const unsigned ob = __ballot_sync(kFull, cv != -1);
                if (lane == qb >> 5) occ |= ob;
                const int64_t j = static_cast<int64_t>(cv) - n0;
                const bool known = cv >= 0 && j >= 0 && j < nt;
                rbad |= cv >= 0 && !known;
                const unsigned kb = __ballot_sync(kFull, known);
                const int at = ne + __popc(kb & ((1u << lane) - 1u));
                if (known && at < kPlEntCap) sm.ent[at] = q << 8 | sm.s2r[j];
                ne += __popc(kb);
              }
            }
            sm.run[lane] = pl_free_starts(occ, Q, cw, lane);
            rbad = __any_sync(kFull, rbad);
            if (lane == 0) {
              sm.ne = ne;
              sm.rbad = rbad;
            }
          }
          __syncthreads();
          if (sm.rbad) {
            st |= QOT_CAND_BAD_STATE;
            break;
          }
          // ---- the free starts in ascending order, dealt round-robin to the warps
          const int ne = sm.ne;
          for (int wd2 = 0; wd2 < 32 && 32 * wd2 < Q; ++wd2) {
            for (unsigned fb = sm.run[wd2]; fb; fb &= fb - 1u) {
              const int q0 = 32 * wd2 + __ffs(fb) - 1;
              if (seq++ % kCdWarps != w) continue;
              if (lane < kCdMaskWords) ws.mask[lane] = 0u;
              __syncwarp();
              if (ne <= kPlEntCap) pl_ent_mask(a, sm.ent, ne, q0, cw, ws.mask, lane);
              else pv_scan(va, sm, b, n0, p0, p1, q0, cw, ws.mask, lane);
              __syncwarp();
              const int nn = cd_rank(lane < kCdMaskWords ? ws.mask[lane] : 0u, ws.nbr, lane);
              cd_xrow(a, ws.cx, [&] { return lane == 0 ? static_cast<float>(a.freqs[q0]) : a.feat[po * 3 + lane - 1]; },
                      lane);
              const int slot = wseq++ & (kPlRing - 1);
              const int nimp = pa.bound ? nn : 0;         // impact rows count against a bound, all of them
              if (lane == 0) {
                ws.nbr[nn] = kCand;
                PlPending& pp = pw.ring[slot];
                pp.mkey = 0xffffffffu;
                pp.left = 1 + nimp;
                pp.p = static_cast<int>(po);
                pp.q0 = q0;
                ++pw.n_free;
              }
              __syncwarp();
              row(ws.nbr, nn + 1, kCand, nullptr, slot, -1);
              for (int e = 0; e < nimp; ++e) {
                const int r = ws.nbr[e];
                const int m = cd_rank(lane < kCdMaskWords ? sm.adj[r][lane] : 0u, ws.msg, lane);
                if (lane == 0) {
                  ws.msg[m] = kCand;
                  ws.msg[m + 1] = r;
                }
                __syncwarp();
                row(ws.msg, m + 2, r, nullptr, slot, b * kCdMaxN + sm.r2s[r]);
              }
            }
          }
          __syncthreads();                                // the entries and free words are read
        }
        // ---- every placement folded: the block's winner and counts
        if (zc) {
          pl_flush(pa, pw, w, zc, o0, lane);
          zc = 0;
        }
        __syncthreads();
        if (tid == 0) {
          unsigned long long key = 0ull;
          int nf = 0, nfe = 0, bw = -1;
          for (int u = 0; u < kCdWarps; ++u) {
            nf += sm.w[u].n_free;
            nfe += sm.w[u].n_feas;
            if (sm.w[u].key > key) {
              key = sm.w[u].key;
              bw = u;
            }
          }
          sm.key_best = key;
          sm.n_free = nf;
          sm.n_feas = nfe;
          if (bw >= 0)
            for (int o = 0; o < 4; ++o) sm.best[o] = sm.w[bw].best[o];
        }
        __syncthreads();
        // ---- warp 0: the winner's neighbours (for pv_commit) and the demand's outputs; acceptance
        if (w == 0) {
          const unsigned long long key = st ? 0ull : sm.key_best;
          int bp = -1, bq = -1;
          int64_t po = -1, p0 = 0, p1 = 0;
          int cw = 0;
          if (key) {
            const unsigned idx = 0xffffffffu - static_cast<unsigned>(key);
            bp = static_cast<int>(idx >> 10);
            bq = static_cast<int>(idx & 1023u);
            po = o0 + bp;
            p0 = a.link_ptr[po];
            p1 = a.link_ptr[po + 1];
            cw = a.width[po];
            if (lane < kCdMaskWords) sm.wmask[lane] = 0u;
            __syncwarp();
            pv_scan(va, sm, b, n0, p0, p1, bq, cw, sm.wmask, lane);
            cd_xrow(a, ws.cx, [&] { return lane == 0 ? static_cast<float>(a.freqs[bq]) : a.feat[po * 3 + lane - 1]; },
                    lane);
            __syncwarp();
          }
          const bool fatal = st & (kPlFatal | QOT_REST_NO_OPTION);
          // the graph builder refuses a sample over QOT_TG_MAX_NODES lightpaths or QOT_TG_MAX_CHANNELS channels
          const bool full = key && (sm.n_tot >= kCdMaxN || sm.n_chan + (p1 - p0) * cw > QOT_TG_MAX_CHANNELS);
          const bool acc = key && !full;
          int first = INT_MAX;                            // the accepted lightpath's first channel
          for (int64_t e = p0 + lane; acc && e < p1; e += 32) first = min(first, a.links[e] * Q + bq);
          first = __reduce_min_sync(kFull, first);
          if (i < MC) {
            if (lane < QOT_OUT) a.out[k * QOT_OUT + lane] = key ? sm.best[lane] : nan;
            if (lane == 0) {
              ra.cut_node[k] = v;
              a.status[k] = st | (full ? QOT_PROV_FULL : 0);
              pa.option[k] = bp;
              pa.q0[k] = bq;
              pa.margin[k] = key ? sm.best[3] : nan;
              pa.n_free[k] = fatal ? 0 : sm.n_free;
              pa.n_feasible[k] = fatal ? 0 : sm.n_feas;
            }
          }
          if (lane == 0) {
            sm.acc = acc;
            sm.c_po = po;
            sm.c_q0 = bq;
            sm.c_key = first;
          }
        }
        __syncthreads();
        if (!sm.acc) continue;
        pv_commit(va, sm, b, n0, tid);
        if (tid == 0) {                                   // the restored lightpath keeps its conn_id
          sm.conn[sm.s2r[sm.n_tot - 1]] = rs.c_conn;
          ++rs.n_rest;
        }
      }
    // ---- the end state: every rank's row through the head, its margin against its bound
    __syncthreads();
    const int nt = sm.n_tot;
    if (pa.bound || ra.end_out) {
      const auto flush = [&](int cnt) {
        cd_flush(w, cnt, a.prep, lane);
        if (lane == 0) rs_end_fold(ra, rs, pw, cnt, f);
        __syncwarp();
      };
      for (int r = w; r < nt; r += kCdWarps) {
        const int m = cd_rank(lane < kCdMaskWords ? sm.adj[r][lane] : 0u, ws.msg, lane);
        if (lane == 0) {
          ws.msg[m] = r;
          pw.rtag[zc] = r;
          pw.rnode[zc] = b * kCdMaxN + sm.r2s[r];
        }
        __syncwarp();
        zc = cd_row(ws, zc, ws.msg, m + 1, r, PvX{sm.x, ws.cx, r, a.lut_col}, As, Ad, pw.rout[zc], flush, lane);
      }
      if (zc) {
        flush(zc);
        zc = 0;
      }
    }
    __syncthreads();
    // ---- the scenario's outputs, the unused cut rows and end rows
    if (tid == 0) {
      ra.status[f] = fst | (ncut > MC ? QOT_REST_CUT_OVERFLOW : 0);
      ra.n_cut[f] = ncut;
      ra.n_restored[f] = rs.n_rest;
      ra.end_margin[f] = pa.bound && nt ? pl_unkey(rs.e_mkey) : nan;
      ra.n_below[f] = pa.bound ? rs.e_below : 0;
    }
    for (int64_t u = f * MC + min(ncut, MC) + tid; u < (f + 1) * MC; u += kCdThreads) {
      ra.cut_node[u] = -1;
      a.status[u] = 0;
      pa.option[u] = pa.q0[u] = -1;
      pa.margin[u] = nan;
      pa.n_free[u] = pa.n_feasible[u] = 0;
      for (int o = 0; o < QOT_OUT; ++o) a.out[u * QOT_OUT + o] = nan;
    }
    if (ra.end_conn) {
      for (int r = tid; r < kCdMaxN; r += kCdThreads) ra.end_conn[f * kCdMaxN + r] = r < nt ? sm.conn[r] : -1;
      for (int u = nt * QOT_OUT + tid; u < kCdMaxN * QOT_OUT; u += kCdThreads)
        ra.end_out[f * kCdMaxN * QOT_OUT + u] = nan;
    }
  }
}

static int cfg_check(const qot_lp_graph_cfg_t* cfg, const char* who) {
  QOT_REQUIRE(cfg, "%s: null cfg", who);
  QOT_REQUIRE(cfg->F > 0 && cfg->L > 0 && cfg->Q > 0 && cfg->L <= 65535 && cfg->Q <= 65535 &&
                  static_cast<int64_t>(cfg->L) * cfg->Q < (1ll << 30), "%s: bad tensor extents", who);
  QOT_REQUIRE(cfg->i_conn >= 0 && cfg->i_conn < cfg->F, "%s: conn_id row out of range", who);
  return QOT_OK;
}

// the checks every network-state entry point makes first: cfg, the sizes (the state's, max_impact and the query's,
// query_ok), the head's table, the flag column
static int cd_check_args(const char* who, const qot_lp_state_t& st, bool query_ok, const float* prepared,
                         int32_t is_lut_index, int32_t max_impact) {
  if (int rc = cfg_check(&st.cfg, who)) return rc;
  QOT_REQUIRE(st.S >= 0 && st.N >= 0 && st.N < INT_MAX && st.E >= 0 && max_impact >= 0 && query_ok, "%s: bad size",
              who);
  QOT_REQUIRE(prepared && (reinterpret_cast<uintptr_t>(prepared) & 15) == 0, "%s: prepared must be 16-byte aligned",
              who);
  QOT_REQUIRE(is_lut_index >= 0 && is_lut_index < kF, "%s: is_lut_index out of range", who);
  return QOT_OK;
}

// the opt-in to kSmem bytes of dynamic shared memory, once per device and kernel
template <auto kKernel, int kSmem>
static int cd_smem_opt_in() {
  static std::atomic<unsigned long long> done{0};
  return once_per_device(done, [] {
    QOT_CUDA(cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    return static_cast<int>(QOT_OK);
  });
}

// the state half of CdArgs (with the head's table and the output width), after the null-state check
static int cd_state_args(const char* who, CdArgs& a, const qot_lp_state_t& st, const float* prepared,
                         int32_t is_lut_index, int32_t max_impact) {
  QOT_REQUIRE(st.S == 0 ||
                  (st.freqs && st.x && st.node_ptr && st.rowptr && st.chan_node && (st.E == 0 || st.edge_index)),
              "%s: null state array", who);
  a.cfg = st.cfg;
  a.S = st.S; a.N = st.N; a.E = st.E;
  a.freqs = st.freqs; a.x = st.x; a.node_ptr = st.node_ptr; a.rowptr = st.rowptr;
  a.edst = st.edge_index ? st.edge_index + st.E : nullptr;
  a.chan_node = st.chan_node;
  a.prep = prepared; a.lut_col = is_lut_index; a.max_impact = max_impact;
  return QOT_OK;
}

// the checks the three change entry points make before their empty-query return (sizes_ok: their own sizes), then the
// change half of CdArgs
static int cd_change_args(const char* who, CdArgs& a, const qot_lp_state_t* st, const qot_lp_changes_t* c,
                          bool sizes_ok, const float* prepared, int32_t is_lut_index, int32_t max_impact) {
  QOT_REQUIRE(st && c, "%s: null state or changes descriptor", who);
  if (int rc = cd_check_args(who, *st, c->K >= 0 && c->n_links >= 0 && sizes_ok, prepared, is_lut_index, max_impact))
    return rc;
  a.K = c->K; a.n_links = c->n_links;
  a.node = c->node;
  a.sample = c->sample; a.link_ptr = c->link_ptr; a.links = c->links; a.q0 = c->q0; a.width = c->width;
  a.feat = c->feat;
  return QOT_OK;
}

// the checks the two demand entry points make before their empty-query return, then the demand half of PlArgs
static int pl_demand_args(const char* who, PlArgs& pa, const qot_lp_state_t* st, const qot_lp_demands_t* d,
                          int32_t metric, int32_t maximize, int32_t policy, const float* prepared, int32_t is_lut_index,
                          int32_t max_impact) {
  QOT_REQUIRE(st && d, "%s: null state or demands descriptor", who);
  if (int rc = cd_check_args(who, *st, d->D >= 0 && d->P >= 0 && d->n_links >= 0, prepared, is_lut_index, max_impact))
    return rc;
  QOT_REQUIRE(st->cfg.Q <= QOT_PLACE_MAX_SLOTS, "%s: Q = %d over QOT_PLACE_MAX_SLOTS", who, st->cfg.Q);
  QOT_REQUIRE(metric >= 0 && metric < QOT_OUT, "%s: metric must be an output column 0..2", who);
  QOT_REQUIRE(policy == QOT_PLACE_FIRST_FIT || policy == QOT_PLACE_BEST_QOT || policy == QOT_PLACE_MAX_MARGIN,
              "%s: unknown policy %d", who, policy);
  CdArgs& a = pa.c;
  a.K = d->D; a.n_links = d->n_links;
  a.node = nullptr;
  a.sample = d->sample; a.link_ptr = d->link_ptr; a.links = d->links; a.q0 = nullptr; a.width = d->width;
  a.feat = d->feat;
  a.impact_kind = nullptr;
  pa.P = d->P; pa.opt_ptr = d->opt_ptr; pa.own_bound = d->own_bound;
  pa.metric = metric; pa.maximize = maximize != 0; pa.policy = policy;
  return QOT_OK;
}

// qot_lightpath_candidates (kMove = false) and qot_lightpath_reconfigure (kMove = true)
template <bool kMove>
static int cd_launch(const char* who, const qot_lp_state_t* state, const qot_lp_changes_t* changes,
                     const float* prepared, int32_t is_lut_index, int32_t max_impact, float* out, int32_t* status,
                     int32_t* n_impact, int64_t* impact_node, int8_t* impact_kind, float* impact_out, void* stream) {
  CdArgs a;
  if (int rc = cd_change_args(who, a, state, changes, true, prepared, is_lut_index, max_impact)) return rc;
  const qot_lp_changes_t& c = *changes;
  if (c.K == 0) return QOT_OK;
  QOT_REQUIRE(c.sample && c.link_ptr && c.q0 && c.width && c.feat && out && status && n_impact &&
                  (c.n_links == 0 || c.links) && (max_impact == 0 || (impact_node && impact_out)) && (!kMove || c.node),
              "%s: null candidate or output array", who);
  if (int rc = cd_state_args(who, a, *state, prepared, is_lut_index, max_impact)) return rc;
  constexpr int smem = static_cast<int>(sizeof(CdSmem));
  if (int rc = cd_smem_opt_in<lp_candidate_kernel<kMove>, smem>()) return rc;
  a.out = out; a.status = status; a.n_impact = n_impact; a.impact_node = impact_node;
  a.impact_kind = max_impact ? impact_kind : nullptr; a.impact_out = impact_out;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, cdiv(c.K, kCdWarps)));
  lp_candidate_kernel<kMove><<<grid, kCdThreads, smem, static_cast<cudaStream_t>(stream)>>>(a);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

// qot_lightpath_protect's additions: the protect flags and the backup outputs
struct PtOut {
  const uint8_t* protect;
  int32_t *option, *q0;
  float *out, *margin;
  int32_t *n_free, *n_feasible, *status, *n_impact;
  int64_t *conn_id, *impact_conn;
  float* impact_out;
};

// qot_lightpath_provision (rel = pt = null), qot_lightpath_traffic (pt = null) and qot_lightpath_protect (rel = null):
// the checks, the copy of chan_node and the launch
static int pv_launch(const char* who, const qot_lp_state_t* state, const qot_lp_demands_t* demands,
                     const int64_t* order, const int64_t* sample_ptr, const float* bound, int32_t metric,
                     int32_t maximize, int32_t policy, const float* prepared, int32_t is_lut_index, int32_t max_impact,
                     int32_t* chan_work, float* bound_work, int32_t* option, int32_t* q0, float* out, float* margin,
                     int32_t* n_free, int32_t* n_feasible, int32_t* status, int32_t* n_impact, int64_t* conn_id,
                     int64_t* impact_conn, float* impact_out, const qot_lp_releases_t* rel, const int64_t* rel_order,
                     const int64_t* rel_ptr, int32_t* rel_status, int64_t* rel_conn_id, int32_t* rel_n_impact,
                     int64_t* rel_impact_conn, float* rel_impact_out, float* rel_margin, cudaStream_t stream,
                     const PtOut* pt = nullptr) {
  PvArgs va;
  PlArgs& pa = va.p;
  CdArgs& a = pa.c;
  if (int rc = pl_demand_args(who, pa, state, demands, metric, maximize, policy, prepared, is_lut_index, max_impact))
    return rc;
  const qot_lp_state_t& st = *state;
  const qot_lp_demands_t& d = *demands;
  const int64_t NR = rel ? rel->R : 0;
  QOT_REQUIRE(NR >= 0, "%s: bad release count", who);
  QOT_REQUIRE(!pt || st.cfg.L <= QOT_TG_MAX_LINKS, "%s: L = %d over QOT_TG_MAX_LINKS (the link bitmaps)", who,
              st.cfg.L);
  if (d.D == 0 && NR == 0) return QOT_OK;
  QOT_REQUIRE(!pt || (pt->option && pt->q0 && pt->out && pt->margin && pt->n_free && pt->n_feasible && pt->status &&
                      pt->n_impact && pt->conn_id && (max_impact == 0 || (pt->impact_conn && pt->impact_out))),
              "%s: null backup output array", who);
  QOT_REQUIRE(d.D == 0 || (d.sample && order && d.opt_ptr && d.link_ptr &&
                           (d.P == 0 || (d.width && d.feat && d.own_bound)) && (d.n_links == 0 || d.links)),
              "%s: null demand or grouping array", who);
  QOT_REQUIRE(sample_ptr, "%s: null demand or grouping array", who);
  QOT_REQUIRE(d.D == 0 || (option && q0 && out && margin && n_free && n_feasible && status && n_impact && conn_id &&
                           (max_impact == 0 || (impact_conn && impact_out))), "%s: null output array", who);
  QOT_REQUIRE((st.S == 0 || chan_work) && (!bound || st.S == 0 || bound_work) && (st.N == 0 || st.conn_ids),
              "%s: null work or conn_ids array", who);
  if (NR > 0) {
    QOT_REQUIRE(rel->sample && rel->before && rel->demand && rel->conn_id && rel_order && rel_ptr,
                "%s: null release or release grouping array", who);
    QOT_REQUIRE(rel_status && rel_conn_id && rel_n_impact && rel_margin &&
                    (max_impact == 0 || (rel_impact_conn && rel_impact_out)), "%s: null release output array", who);
  }
  if (int rc = cd_state_args(who, a, st, prepared, is_lut_index, max_impact)) return rc;
  constexpr int smem = static_cast<int>(sizeof(PvSmem)), pt_smem = static_cast<int>(sizeof(PtSmem));
  if (int rc = pt        ? cd_smem_opt_in<lp_provision_kernel<false, true>, pt_smem>()
               : NR > 0  ? cd_smem_opt_in<lp_provision_kernel<true>, smem>()
                         : cd_smem_opt_in<lp_provision_kernel<false>, smem>())
    return rc;
  if (st.S > 0)
    QOT_CUDA(cudaMemcpyAsync(chan_work, st.chan_node, static_cast<size_t>(st.S) * st.cfg.L * st.cfg.Q * sizeof(int32_t),
                             cudaMemcpyDeviceToDevice, stream));
  a.chan_node = chan_work;
  a.out = out; a.status = status; a.n_impact = n_impact; a.impact_node = impact_conn; a.impact_out = impact_out;
  pa.bound = bound ? bound_work : nullptr;
  pa.option = option; pa.q0 = q0; pa.margin = margin; pa.n_free = n_free; pa.n_feasible = n_feasible;
  pa.all_out = nullptr; pa.all_margin = nullptr;
  va.order = order; va.sample_ptr = sample_ptr; va.conn_ids = st.conn_ids; va.bound = bound;
  va.chan_work = chan_work; va.bound_work = bound ? bound_work : nullptr; va.conn_id = conn_id;
  va.rel = NR > 0 ? *rel : qot_lp_releases_t{0, nullptr, nullptr, nullptr, nullptr};
  va.rel_order = rel_order; va.rel_ptr = NR > 0 ? rel_ptr : nullptr;
  va.rel_status = rel_status; va.rel_conn_id = rel_conn_id; va.rel_n_impact = rel_n_impact;
  va.rel_impact_conn = rel_impact_conn; va.rel_impact_out = rel_impact_out; va.rel_margin = rel_margin;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, std::max<int64_t>(1, st.S)));
  if (pt) {
    PtArgs ta;
    static_cast<PvArgs&>(ta) = va;
    ta.bk = va;
    ta.bk.p.c.out = pt->out; ta.bk.p.c.status = pt->status; ta.bk.p.c.n_impact = pt->n_impact;
    ta.bk.p.c.impact_node = pt->impact_conn; ta.bk.p.c.impact_out = pt->impact_out;
    ta.bk.p.option = pt->option; ta.bk.p.q0 = pt->q0; ta.bk.p.margin = pt->margin;
    ta.bk.p.n_free = pt->n_free; ta.bk.p.n_feasible = pt->n_feasible;
    ta.bk.conn_id = pt->conn_id;
    ta.protect = pt->protect;
    lp_provision_kernel<false, true><<<grid, kCdThreads, pt_smem, stream>>>(ta);
  } else if (NR > 0) {
    lp_provision_kernel<true><<<grid, kCdThreads, smem, stream>>>(va);
  } else {
    lp_provision_kernel<false><<<grid, kCdThreads, smem, stream>>>(va);
  }
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

// qot_lightpath_restore: the checks and the launch (the kernel copies each scenario's chan_node row itself)
static int rs_launch(const qot_lp_state_t* state, const qot_lp_demands_t* options, const qot_lp_failures_t* failures,
                     int32_t policy, int32_t metric, int32_t maximize, const float* bound, const float* prepared,
                     int32_t is_lut_index, int32_t max_cut, int32_t* chan_work, float* bound_work, int32_t n_blocks,
                     int64_t* cut_node, int32_t* option, int32_t* q0, float* out, float* margin, int32_t* n_free,
                     int32_t* n_feasible, int32_t* cut_status, int32_t* status, int32_t* n_cut, int32_t* n_restored,
                     float* end_margin, int32_t* n_below, int64_t* end_conn, float* end_out, cudaStream_t stream) {
  const char* who = "qot_lightpath_restore";
  RsArgs ra;
  PvArgs& va = ra.v;
  PlArgs& pa = va.p;
  CdArgs& a = pa.c;
  QOT_REQUIRE(failures, "%s: null failures descriptor", who);
  if (int rc = pl_demand_args(who, pa, state, options, metric, maximize, policy, prepared, is_lut_index, 0)) return rc;
  const qot_lp_state_t& st = *state;
  const qot_lp_demands_t& d = *options;
  const qot_lp_failures_t& fl = *failures;
  QOT_REQUIRE(fl.F >= 0 && fl.n_links >= 0 && max_cut >= 0 && n_blocks >= 1, "%s: bad size", who);
  QOT_REQUIRE(d.D == st.N, "%s: the options hold %lld demands, the state %lld nodes (one demand per node)", who,
              static_cast<long long>(d.D), static_cast<long long>(st.N));
  if (fl.F == 0) return QOT_OK;
  QOT_REQUIRE(fl.sample && fl.link_ptr && (fl.n_links == 0 || fl.links), "%s: null failure array", who);
  QOT_REQUIRE(d.D == 0 || (d.sample && d.opt_ptr && d.link_ptr && (d.P == 0 || (d.width && d.feat && d.own_bound)) &&
                           (d.n_links == 0 || d.links)),
              "%s: null option array", who);
  QOT_REQUIRE(status && n_cut && n_restored && end_margin && n_below && !end_conn == !end_out &&
                  (max_cut == 0 || (cut_node && option && q0 && out && margin && n_free && n_feasible && cut_status)),
              "%s: null output array", who);
  QOT_REQUIRE(chan_work && (!bound || bound_work) && (st.N == 0 || st.conn_ids), "%s: null work or conn_ids array",
              who);
  if (int rc = cd_state_args(who, a, st, prepared, is_lut_index, 0)) return rc;
  constexpr int smem = static_cast<int>(sizeof(RsSmem));
  if (int rc = cd_smem_opt_in<lp_restore_kernel, smem>()) return rc;
  a.chan_node = chan_work;
  a.out = out; a.status = cut_status; a.n_impact = nullptr; a.impact_node = nullptr; a.impact_out = nullptr;
  pa.bound = bound ? bound_work : nullptr;
  pa.option = option; pa.q0 = q0; pa.margin = margin; pa.n_free = n_free; pa.n_feasible = n_feasible;
  pa.all_out = nullptr; pa.all_margin = nullptr;
  va = PvArgs{pa, nullptr, nullptr, st.conn_ids, bound, chan_work, bound ? bound_work : nullptr, nullptr,
              qot_lp_releases_t{0, nullptr, nullptr, nullptr, nullptr}, nullptr, nullptr, nullptr, nullptr, nullptr,
              nullptr, nullptr, nullptr};
  ra.chan_node = st.chan_node;
  ra.fail = fl;
  ra.max_cut = max_cut;
  ra.cut_node = cut_node; ra.status = status; ra.n_cut = n_cut; ra.n_restored = n_restored;
  ra.end_margin = end_margin; ra.n_below = n_below; ra.end_conn = end_conn; ra.end_out = end_out;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(n_blocks, fl.F));
  lp_restore_kernel<<<grid, kCdThreads, smem, stream>>>(ra);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

}  // namespace qot

using namespace qot;

extern "C" int qot_lightpath_channel_map(const float* data, int64_t S, const qot_lp_graph_cfg_t* cfg,
                                         const int64_t* node_ptr, const int64_t* conn_ids, int64_t N,
                                         int32_t* chan_node, int32_t* status, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (int rc = cfg_check(cfg, "qot_lightpath_channel_map")) return rc;
  QOT_REQUIRE(S >= 0 && N >= 0 && N < INT_MAX, "qot_lightpath_channel_map: bad sample or node count");
  QOT_REQUIRE(S == 0 || (data && node_ptr && chan_node && (N == 0 || conn_ids)),
              "qot_lightpath_channel_map: null argument");
  if (S == 0) return QOT_OK;
  lp_channel_map_kernel<<<static_cast<unsigned>(S), kCmThreads, 0, stream>>>(data, *cfg, node_ptr, conn_ids, N,
                                                                              chan_node, status);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

extern "C" int qot_lightpath_candidates(const qot_lp_state_t* state, const qot_lp_changes_t* cands,
                                        const float* prepared, int32_t is_lut_index, int32_t max_impact, float* out,
                                        int32_t* status, int32_t* n_impact, int64_t* impact_node, float* impact_out,
                                        void* stream) {
  return cd_launch<false>("qot_lightpath_candidates", state, cands, prepared, is_lut_index, max_impact, out, status,
                          n_impact, impact_node, nullptr, impact_out, stream);
}

extern "C" int qot_lightpath_reconfigure(const qot_lp_state_t* state, const qot_lp_changes_t* changes,
                                         const float* prepared, int32_t is_lut_index, int32_t max_impact, float* out,
                                         int32_t* status, int32_t* n_impact, int64_t* impact_node,
                                         int8_t* impact_kind, float* impact_out, void* stream) {
  return cd_launch<true>("qot_lightpath_reconfigure", state, changes, prepared, is_lut_index, max_impact, out, status,
                         n_impact, impact_node, impact_kind, impact_out, stream);
}

extern "C" int qot_lightpath_change_sets(const qot_lp_state_t* state, const qot_lp_changes_t* changes, int64_t G,
                                         const int64_t* set_ptr, const float* prepared, int32_t is_lut_index,
                                         int32_t max_impact, float* out, int32_t* status, int32_t* set_status,
                                         int32_t* n_impact, int64_t* impact_node, int8_t* impact_kind,
                                         float* impact_out, void* stream) {
  const char* who = "qot_lightpath_change_sets";
  CsArgs ca;
  CdArgs& a = ca.c;
  if (int rc = cd_change_args(who, a, state, changes, G >= 0, prepared, is_lut_index, max_impact)) return rc;
  const qot_lp_changes_t& c = *changes;
  if (G == 0 && c.K == 0) return QOT_OK;
  QOT_REQUIRE(set_ptr && (G == 0 || (set_status && n_impact && (max_impact == 0 || (impact_node && impact_out)))),
              "%s: null set or set output array", who);
  QOT_REQUIRE(c.K == 0 || (c.node && c.sample && c.link_ptr && c.q0 && c.width && c.feat && out && status &&
                           (c.n_links == 0 || c.links)),
              "%s: null change or change output array", who);
  if (int rc = cd_state_args(who, a, *state, prepared, is_lut_index, max_impact)) return rc;
  constexpr int smem = static_cast<int>(sizeof(CsSmem));
  if (int rc = cd_smem_opt_in<lp_change_set_kernel, smem>()) return rc;
  a.out = nullptr; a.status = set_status; a.n_impact = n_impact; a.impact_node = impact_node;
  a.impact_kind = max_impact ? impact_kind : nullptr; a.impact_out = impact_out;
  ca.G = G; ca.set_ptr = set_ptr; ca.chg_out = out; ca.chg_status = status;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, std::max<int64_t>(1, cdiv(G, kCdWarps))));
  lp_change_set_kernel<<<grid, kCdThreads, smem, static_cast<cudaStream_t>(stream)>>>(ca);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

extern "C" int qot_lightpath_placements(const qot_lp_state_t* state, const qot_lp_demands_t* demands,
                                        const float* bound, int32_t metric, int32_t maximize, int32_t policy,
                                        const float* prepared, int32_t is_lut_index, int32_t max_impact,
                                        int32_t* option, int32_t* q0, float* out, float* margin, int32_t* n_free,
                                        int32_t* n_feasible, int32_t* status, int32_t* n_impact,
                                        int64_t* impact_node, float* impact_out, float* all_out, float* all_margin,
                                        void* stream) {
  const char* who = "qot_lightpath_placements";
  PlArgs pa;
  CdArgs& a = pa.c;
  if (int rc = pl_demand_args(who, pa, state, demands, metric, maximize, policy, prepared, is_lut_index, max_impact))
    return rc;
  const qot_lp_demands_t& d = *demands;
  if (d.D == 0) return QOT_OK;
  QOT_REQUIRE(d.sample && d.opt_ptr && d.link_ptr && (d.P == 0 || (d.width && d.feat && d.own_bound)) &&
                  (d.n_links == 0 || d.links),
              "%s: null demand array", who);
  QOT_REQUIRE(option && q0 && out && margin && n_free && n_feasible && status && n_impact &&
                  (max_impact == 0 || (impact_node && impact_out)) && (!all_out == !all_margin),
              "%s: null output array", who);
  if (int rc = cd_state_args(who, a, *state, prepared, is_lut_index, max_impact)) return rc;
  constexpr int smem = static_cast<int>(sizeof(PlSmem));
  if (int rc = cd_smem_opt_in<lp_placement_kernel, smem>()) return rc;
  a.out = out; a.status = status; a.n_impact = n_impact; a.impact_node = impact_node; a.impact_out = impact_out;
  pa.bound = bound;
  pa.option = option; pa.q0 = q0; pa.margin = margin; pa.n_free = n_free; pa.n_feasible = n_feasible;
  pa.all_out = all_out; pa.all_margin = all_margin;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, cdiv(d.D, kCdWarps)));
  lp_placement_kernel<<<grid, kCdThreads, smem, static_cast<cudaStream_t>(stream)>>>(pa);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

extern "C" int qot_lightpath_provision(const qot_lp_state_t* state, const qot_lp_demands_t* demands,
                                       const int64_t* order, const int64_t* sample_ptr, const float* bound,
                                       int32_t metric, int32_t maximize, int32_t policy, const float* prepared,
                                       int32_t is_lut_index, int32_t max_impact, int32_t* chan_work, float* bound_work,
                                       int32_t* option, int32_t* q0, float* out, float* margin, int32_t* n_free,
                                       int32_t* n_feasible, int32_t* status, int32_t* n_impact, int64_t* conn_id,
                                       int64_t* impact_conn, float* impact_out, void* stream) {
  return pv_launch("qot_lightpath_provision", state, demands, order, sample_ptr, bound, metric, maximize, policy,
                   prepared, is_lut_index, max_impact, chan_work, bound_work, option, q0, out, margin, n_free,
                   n_feasible, status, n_impact, conn_id, impact_conn, impact_out, nullptr, nullptr, nullptr, nullptr,
                   nullptr, nullptr, nullptr, nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

extern "C" int qot_lightpath_traffic(const qot_lp_state_t* state, const qot_lp_demands_t* demands,
                                     const int64_t* order, const int64_t* sample_ptr, const float* bound,
                                     int32_t metric, int32_t maximize, int32_t policy, const float* prepared,
                                     int32_t is_lut_index, int32_t max_impact, int32_t* chan_work, float* bound_work,
                                     int32_t* option, int32_t* q0, float* out, float* margin, int32_t* n_free,
                                     int32_t* n_feasible, int32_t* status, int32_t* n_impact, int64_t* conn_id,
                                     int64_t* impact_conn, float* impact_out, const qot_lp_releases_t* releases,
                                     const int64_t* rel_order, const int64_t* rel_ptr, int32_t* rel_status,
                                     int64_t* rel_conn_id, int32_t* rel_n_impact, int64_t* rel_impact_conn,
                                     float* rel_impact_out, float* rel_margin, void* stream) {
  const char* who = "qot_lightpath_traffic";
  QOT_REQUIRE(releases, "%s: null releases descriptor", who);
  return pv_launch(who, state, demands, order, sample_ptr, bound, metric, maximize, policy, prepared, is_lut_index,
                   max_impact, chan_work, bound_work, option, q0, out, margin, n_free, n_feasible, status, n_impact,
                   conn_id, impact_conn, impact_out, releases, rel_order, rel_ptr, rel_status, rel_conn_id,
                   rel_n_impact, rel_impact_conn, rel_impact_out, rel_margin, static_cast<cudaStream_t>(stream));
}

extern "C" int qot_lightpath_protect(const qot_lp_state_t* state, const qot_lp_demands_t* demands,
                                     const int64_t* order, const int64_t* sample_ptr, const float* bound,
                                     int32_t metric, int32_t maximize, int32_t policy, const float* prepared,
                                     int32_t is_lut_index, int32_t max_impact, int32_t* chan_work, float* bound_work,
                                     int32_t* option, int32_t* q0, float* out, float* margin, int32_t* n_free,
                                     int32_t* n_feasible, int32_t* status, int32_t* n_impact, int64_t* conn_id,
                                     int64_t* impact_conn, float* impact_out, const uint8_t* protect,
                                     int32_t* backup_option, int32_t* backup_q0, float* backup_out,
                                     float* backup_margin, int32_t* backup_n_free, int32_t* backup_n_feasible,
                                     int32_t* backup_status, int32_t* backup_n_impact, int64_t* backup_conn_id,
                                     int64_t* backup_impact_conn, float* backup_impact_out, void* stream) {
  const PtOut pt{protect, backup_option, backup_q0, backup_out, backup_margin, backup_n_free, backup_n_feasible,
                 backup_status, backup_n_impact, backup_conn_id, backup_impact_conn, backup_impact_out};
  return pv_launch("qot_lightpath_protect", state, demands, order, sample_ptr, bound, metric, maximize, policy,
                   prepared, is_lut_index, max_impact, chan_work, bound_work, option, q0, out, margin, n_free,
                   n_feasible, status, n_impact, conn_id, impact_conn, impact_out, nullptr, nullptr, nullptr, nullptr,
                   nullptr, nullptr, nullptr, nullptr, nullptr, static_cast<cudaStream_t>(stream), &pt);
}

extern "C" int qot_lightpath_restore(const qot_lp_state_t* state, const qot_lp_demands_t* options,
                                     const qot_lp_failures_t* failures, int32_t policy, int32_t metric,
                                     int32_t maximize, const float* bound, const float* prepared, int32_t is_lut_index,
                                     int32_t max_cut, int32_t* chan_work, float* bound_work, int32_t n_blocks,
                                     int64_t* cut_node, int32_t* option, int32_t* q0, float* out, float* margin,
                                     int32_t* n_free, int32_t* n_feasible, int32_t* cut_status, int32_t* status,
                                     int32_t* n_cut, int32_t* n_restored, float* end_margin, int32_t* n_below,
                                     int64_t* end_conn, float* end_out, void* stream) {
  return rs_launch(state, options, failures, policy, metric, maximize, bound, prepared, is_lut_index, max_cut,
                   chan_work, bound_work, n_blocks, cut_node, option, q0, out, margin, n_free, n_feasible, cut_status,
                   status, n_cut, n_restored, end_margin, n_below, end_conn, end_out,
                   static_cast<cudaStream_t>(stream));
}
