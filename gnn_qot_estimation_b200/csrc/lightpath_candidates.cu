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

__global__ void __launch_bounds__(kCdThreads, 1) lp_provision_kernel(const __grid_constant__ PvArgs va) {
  const PlArgs& pa = va.p;
  const CdArgs& a = pa.c;
  PvSmem& sm = *reinterpret_cast<PvSmem*>(cd_smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = sm.cd.w[w];
  PlWarpSmem& pw = sm.w[w];
  float As[kF], Ad[kF];
  cd_head_prologue(a.prep, As, Ad, tid);
  if (tid == 0) sm.n_valid = 0ull;
  // ---- the grouping, checked whole by every block: sample_ptr non-decreasing from 0; order[i] a demand of the sample
  // whose range holds i, ascending within the range; the ranges hold every demand with a sample in [0, S).  Otherwise
  // no demand is provisioned: every output says PROV_BAD_GROUPING, each written by exactly one thread of the grid.
  const int64_t S = a.S, D = a.K;
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
  const int64_t gt = static_cast<int64_t>(blockIdx.x) * kCdThreads + tid;
  const int64_t gs = static_cast<int64_t>(gridDim.x) * kCdThreads;
  if (bad) {
    for (int64_t d = gt; d < D; d += gs) pv_empty(va, d, QOT_PROV_BAD_GROUPING, 0, 1);
    return;
  }
  for (int64_t d = gt; d < D; d += gs)
    if (a.sample[d] < 0 || a.sample[d] >= S) pv_empty(va, d, QOT_CAND_BAD_SAMPLE, 0, 1);
  const float nan = __int_as_float(0x7fc00000);
  int zc = 0;                                             // rows staged in this warp's head buffer
  for (int64_t s = blockIdx.x; s < S; s += gridDim.x) {
    const int64_t i0 = va.sample_ptr[s], i1 = va.sample_ptr[s + 1];
    if (i0 == i1) continue;
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
    for (int64_t i = i0; i < i1; ++i) {
      const int64_t d = va.order[i];
      const int64_t o0 = pa.opt_ptr[d], o1 = pa.opt_ptr[d + 1];
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
      for (int64_t po = o0; st == 0 && po < o1; ++po) {
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
            if (lane == 0) a.impact_node[d * MI + k] = sm.conn[r];
            const int m = cd_rank(lane < kCdMaskWords ? sm.adj[r][lane] : 0u, ws.msg, lane);
            if (lane == 0) {
              ws.msg[m] = kCand;
              ws.msg[m + 1] = r;
            }
            __syncwarp();
            row(ws.msg, m + 2, r, a.impact_out + (d * MI + k) * QOT_OUT, -1, -1);
          }
        }
        if (st & kPlFatal) {
          pv_empty(va, d, st, lane, 32);
          if (lane == 0) sm.acc = 0;
        } else {
          cd_clear_impact(a, d, rows, MI, nullptr, lane, 32);
          // the graph builder refuses a sample over QOT_TG_MAX_NODES lightpaths or QOT_TG_MAX_CHANNELS channels
          const bool full = key && (sm.n_tot >= kCdMaxN || sm.n_chan + (p1 - p0) * cw > QOT_TG_MAX_CHANNELS);
          const bool acc = key && !full;
          int first = INT_MAX;                            // the accepted lightpath's first channel
          for (int64_t e = p0 + lane; acc && e < p1; e += 32) first = min(first, a.links[e] * Q + bq);
          first = __reduce_min_sync(kFull, first);
          if (lane < QOT_OUT) a.out[d * QOT_OUT + lane] = key ? sm.best[lane] : nan;
          if (lane == 0) {
            a.status[d] = st | (cnt > MI ? QOT_CAND_IMPACT_OVERFLOW : 0) | (full ? QOT_PROV_FULL : 0);
            a.n_impact[d] = cnt;
            pa.option[d] = bp;
            pa.q0[d] = bq;
            pa.margin[d] = key ? sm.best[3] : nan;
            pa.n_free[d] = sm.n_free;
            pa.n_feasible[d] = sm.n_feas;
            va.conn_id[d] = acc ? sm.top + 1 : -1;
            sm.acc = acc;
            sm.c_po = po;
            sm.c_q0 = bq;
            sm.c_key = first;
          }
        }
      }
      __syncthreads();
      if (!sm.acc) continue;
      pv_commit(va, sm, s, n0, tid);
    }
  }
  if (zc) pl_flush(pa, pw, w, zc, 0, lane);
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
                                       int64_t* impact_conn, float* impact_out, void* stream_) {
  const char* who = "qot_lightpath_provision";
  PvArgs va;
  PlArgs& pa = va.p;
  CdArgs& a = pa.c;
  if (int rc = pl_demand_args(who, pa, state, demands, metric, maximize, policy, prepared, is_lut_index, max_impact))
    return rc;
  const qot_lp_state_t& st = *state;
  const qot_lp_demands_t& d = *demands;
  if (d.D == 0) return QOT_OK;
  QOT_REQUIRE(d.sample && order && sample_ptr && d.opt_ptr && d.link_ptr &&
                  (d.P == 0 || (d.width && d.feat && d.own_bound)) && (d.n_links == 0 || d.links),
              "%s: null demand or grouping array", who);
  QOT_REQUIRE(option && q0 && out && margin && n_free && n_feasible && status && n_impact && conn_id &&
                  (max_impact == 0 || (impact_conn && impact_out)), "%s: null output array", who);
  QOT_REQUIRE((st.S == 0 || chan_work) && (!bound || st.S == 0 || bound_work) && (st.N == 0 || st.conn_ids),
              "%s: null work or conn_ids array", who);
  if (int rc = cd_state_args(who, a, st, prepared, is_lut_index, max_impact)) return rc;
  constexpr int smem = static_cast<int>(sizeof(PvSmem));
  if (int rc = cd_smem_opt_in<lp_provision_kernel, smem>()) return rc;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
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
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, std::max<int64_t>(1, st.S)));
  lp_provision_kernel<<<grid, kCdThreads, smem, stream>>>(va);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}
