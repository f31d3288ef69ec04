// LightpathGNN candidate QoT: a candidate lightpath evaluated against a resident network state without rebuilding
// the state's graph.
//
// Semantics: candidate k names a sample s_k of the state, a path (link indices), a contiguous slot range
// [q0_k, q0_k + width_k) used on every link of the path and its raw feature vector (freq, mod_order, num_spans,
// path_len).  sample' is sample s_k with the candidate written into every channel of its path and slot range (a new
// conn_id, osnr = snr = ber = -1).  In sample''s lightpath graph (to_graph's construction):
//   out[k]           = the eval-mode forward with the flag column one-hot at the candidate's node;
//   impact row i     = the same with the flag at the candidate's i-th neighbour j, neighbours in ascending order of
//                      their node index in the state batch.
// Why no rebuild is needed: the model has one GAT layer and eval-mode BatchNorm is a per-node affine, so a row depends
// only on its node and its in-neighbours.  Inserting the candidate adds exactly the edges candidate <-> j for the
// lightpaths j that share a link with it at 0 < |df| < freq_threshold; every other row of the graph is unchanged.
//
//   lp_channel_map_kernel (once per state): chan_node [S, L, Q] = state-batch node index of the lightpath on each
//     channel, -1 on a free channel (occupancy and conn_id truncation as in to_graph.cu).
//   lp_candidate_kernel: persistent, one warp per candidate.  Validate; scan the chan_node rows of the path's links
//     with the fp64 df test of to_graph.cu, neighbours into a 256-bit per-warp mask (a state sample holds at most
//     QOT_TG_MAX_NODES lightpaths), ranked ascending; then
//       candidate row: query flag 1, the neighbours (flag 0), the appended self loop;
//       impact row j:  query flag 1, j's in-row of the state graph = the destinations of j's out-run in the
//                      source-sorted edge list (self loop dropped, flag 0), the candidate (flag 0), j's self loop.
//     Every z row goes through the warp's 16-row buffer and head_rows16_tf32x3 (the mma.sync head of every-node mode).
//
// Reconfiguration (qot_lightpath_reconfigure, the kMove instantiation): a change is a candidate that also names the
// lightpath j it moves (-1: a plain insertion, bit-identical to the candidate path).  j's old channels count as free,
// its old neighbours (the destinations of its out-run, self loop dropped) go into a second 256-bit mask, and the impact
// rows are the union of both masks, ranked ascending, with kind bits old | new << 1:
//       j's row:         query flag 1, j's new neighbours (flag 0), the appended self loop (none for a teardown);
//       impact row i:    query flag 1, i's state in-row without j (flag 0), j with its new x if i is a new
//                        neighbour (flag 0), i's self loop.
// Every other row of the sample is unchanged, for the same locality reason as a candidate's.
//
// Deterministic: integer mask bits only, fixed message order, no float atomics.  A malformed candidate gets status
// bits and a NaN row; it never faults and never stops the launch.
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

// attention of query node q over msg[0, M) into the next staged z row; the row's outputs go to `dst`
__device__ __forceinline__ int cd_row(CdWarpSmem& ws, int w, int zc, const int* msg, int M, int q, const CdX& xf,
                                      const float (&As)[kF], const float (&Ad)[kF], float* dst,
                                      const float* __restrict__ prep, int lane) {
  float d_q = 0.f;
#pragma unroll
  for (int k = 0; k < kF; ++k) d_q = fmaf(xf(q, k), Ad[k], d_q);
  AttnState st;
  attn_consume(st, msg, M, xf, As, d_q, lane);
  attn_finish<kF>(st, ws.z + zc * kCdZPitch, lane);
  if (lane == 0) ws.orow[zc] = reinterpret_cast<long long>(dst);
  __syncwarp();
  if (++zc == 16) {
    cd_flush(w, 16, prep, lane);
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

// kMove = false: qot_lightpath_candidates; true: qot_lightpath_reconfigure (a.node, a.impact_kind)
template <bool kMove>
__global__ void __launch_bounds__(kCdThreads, 1) lp_candidate_kernel(const __grid_constant__ CdArgs a) {
  CdSmem& sm = cd_smem();
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  CdWarpSmem& ws = sm.w[w];
  for (int i = tid; i < kStHeadFrag4; i += kCdThreads)
    sm.frag[i] = __ldg(reinterpret_cast<const float4*>(a.prep + kOffB1f) + i);
  __syncthreads();
  const float* __restrict__ prep = a.prep;
  const int h = lane & 3;
  float As[kF], Ad[kF];
#pragma unroll
  for (int k = 0; k < kF; ++k) {
    As[k] = __ldg(prep + kOffAsrc + k * kHeads + h);
    Ad[k] = __ldg(prep + kOffAdst + k * kHeads + h);
  }
  const int L = a.cfg.L, Q = a.cfg.Q, MI = a.max_impact;
  const double thr = a.cfg.freq_threshold;
  const float nan = __int_as_float(0x7fc00000);
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
    bool badp = !(p0 >= 0 && p1 > p0 && p1 <= a.n_links) || cw < 1 || c0 < 0 || static_cast<int64_t>(c0) + cw > Q;
    if (kMove && tear) badp = !(p0 >= 0 && p0 <= a.n_links);
    if (!badp)
      for (int64_t e = p0 + lane; e < p1; e += 32) {
        const int l = a.links[e];
        badp |= l < 0 || l >= L;
      }
    if (__any_sync(kFull, badp)) st |= QOT_CAND_BAD_PATH;
    if (kMove && jg != -1 && !(st & QOT_CAND_BAD_SAMPLE) && (jg < a.node_ptr[s] || jg >= a.node_ptr[s + 1]))
      st |= QOT_CAND_BAD_NODE;
    int64_t n0 = 0;
    int n = 0;
    if (st == 0) {
      n0 = a.node_ptr[s];
      const int64_t n1 = a.node_ptr[s + 1];
      if (n0 >= 0 && n1 >= n0 && n1 <= a.N && n1 - n0 <= kCdMaxN) n = static_cast<int>(n1 - n0);
      else st |= QOT_CAND_BAD_STATE;
    }
    const int jm = kMove && st == 0 && jg >= 0 ? static_cast<int>(jg - n0) : -1;   // sample-local; -1 matches no node
    // ---- neighbours: chan_node rows of the path's links, the fp64 df test of to_graph.cu
    if (lane < kCdMaskWords) {
      ws.mask[lane] = 0u;
      if (kMove) ws.omask[lane] = 0u;
    }
    __syncwarp();
    if (st == 0) {
      bool occ = false, bad = false;
      for (int64_t e = p0; e < p1; ++e) {
        const int32_t* __restrict__ row = a.chan_node + (s * L + a.links[e]) * Q;
        for (int q = lane; q < Q; q += 32) {
          const int32_t v = row[q];
          if (v == -1 || (kMove && v == jg)) continue;            // free, or the moved lightpath's own channel
          if (q >= c0 && q < c0 + cw) { occ = true; continue; }
          if (v < -1) continue;                                   // occupied by an unknown lightpath: no edge
          const int64_t j = v - n0;
          if (j < 0 || j >= n) { bad = true; continue; }
          const double fq = a.freqs[q];
          bool hit = false;
          for (int c = c0; c < c0 + cw && !hit; ++c) {
            const double df = fabs(a.freqs[c] - fq);
            hit = df < thr && df > 0.0;
          }
          if (hit) atomicOr(&ws.mask[j >> 5], 1u << (j & 31));
        }
      }
      if (kMove && jm >= 0) {                 // old neighbours: destinations of j's out-run, self loop dropped
        const int64_t r0 = a.rowptr[n0 + jm], r1 = a.rowptr[n0 + jm + 1];
        if (!(r0 >= 0 && r1 >= r0 && r1 <= a.E)) bad = true;
        else
          for (int64_t e = r0 + lane; e < r1; e += 32) {
            const int64_t dg = a.edst[e] - n0;
            if (dg < 0 || dg >= n) bad = true;
            else if (dg != jm) atomicOr(&ws.omask[dg >> 5], 1u << (dg & 31));
          }
      }
      if (__any_sync(kFull, occ)) st |= QOT_CAND_OCCUPIED;
      if (__any_sync(kFull, bad)) st |= QOT_CAND_BAD_STATE;
    }
    __syncwarp();
    if (st & (QOT_CAND_BAD_SAMPLE | QOT_CAND_BAD_PATH | QOT_CAND_OCCUPIED | QOT_CAND_BAD_STATE | QOT_CAND_BAD_NODE)) {
      if (lane < QOT_OUT) a.out[k * QOT_OUT + lane] = nan;
      if (lane == 0) {
        a.status[k] = st;
        a.n_impact[k] = 0;
      }
      for (int i = lane; i < MI; i += 32) a.impact_node[k * MI + i] = -1;
      if (kMove && a.impact_kind)
        for (int i = lane; i < MI; i += 32) a.impact_kind[k * MI + i] = 0;
      for (int i = lane; i < MI * QOT_OUT; i += 32) a.impact_out[k * MI * QOT_OUT + i] = nan;
      continue;
    }
    // ---- neighbours of the new placement ranked ascending: lane t < 8 owns mask word t.  A candidate's impact rows
    // are exactly these; a change's own row takes them from msg and its impact rows are ranked below.
    const unsigned mw = lane < kCdMaskWords ? ws.mask[lane] : 0u;
    int* own = kMove ? ws.msg : ws.nbr;
    const int nn = cd_rank(mw, own, lane);
    if (lane == 0) own[nn] = kCand;                               // the candidate's appended self loop
    // ---- the candidate's x row [freq, is_lut, mod_order, num_spans, path_len]: min-max in fp64 of the float32
    // value, then fp32 (dataset.py's scaling; feat_lo / feat_hi in feat's order)
    if (lane < 4) {
      const double v = static_cast<double>(a.feat[k * 4 + lane]);
      ws.cx[lane == 0 ? 0 : lane + 1] =
          static_cast<float>((v - a.cfg.feat_lo[lane]) / (a.cfg.feat_hi[lane] - a.cfg.feat_lo[lane]));
    }
    if (lane == 4) ws.cx[1] = 1.0f;             // to_graph's is_lut of a lightpath with unknown metrics
    __syncwarp();
    const float* xs = a.x + n0 * kF;
    // ---- candidate row: neighbours (flag 0), then its self loop (flag 1)
    if (kMove && tear) {
      if (lane < QOT_OUT) a.out[k * QOT_OUT + lane] = nan;
    } else {
      zc = cd_row(ws, w, zc, own, nn + 1, kCand, CdX{xs, ws.cx, kCand, a.lut_col}, As, Ad, a.out + k * QOT_OUT,
                  prep, lane);
    }
    int cnt = nn;
    if (kMove) {                             // impact rows of a change: old and new neighbours
      cnt = cd_rank(mw | (lane < kCdMaskWords ? ws.omask[lane] : 0u), ws.nbr, lane);
      __syncwarp();
    }
    if (cnt > MI) st |= QOT_CAND_IMPACT_OVERFLOW;
    // ---- impact rows: neighbour j's in-row (flag 0), the candidate (flag 0), j's self loop (flag 1)
    const int rows = min(cnt, MI);
    for (int i = 0; i < rows; ++i) {
      const int j = ws.nbr[i];
      const int kind = kMove ? static_cast<int>((ws.omask[j >> 5] >> (j & 31) & 1u) |
                                                (ws.mask[j >> 5] >> (j & 31) & 1u) << 1)
                             : 2;            // bit 0: was a neighbour of the moved lightpath, bit 1: is one now
      const int64_t r0 = a.rowptr[n0 + j], r1 = a.rowptr[n0 + j + 1];
      float* dst = a.impact_out + (k * MI + i) * QOT_OUT;
      if (lane == 0) {
        a.impact_node[k * MI + i] = n0 + j;
        if (kMove && a.impact_kind) a.impact_kind[k * MI + i] = static_cast<int8_t>(kind);
      }
      bool bad = !(r0 >= 0 && r1 >= r0 && r1 <= a.E && r1 - r0 <= kCdMaxN);
      int m = 0;
      if (!bad) {
        for (int64_t eb = r0; eb < r1; eb += 32) {
          const int64_t e = eb + lane;
          const int64_t dg = e < r1 ? a.edst[e] - n0 : -1;
          const bool inside = dg >= 0 && dg < n;
          bad |= e < r1 && !inside;
          const bool keep = inside && dg != j && (!kMove || dg != jm);
          const unsigned ball = __ballot_sync(kFull, keep);
          if (keep) ws.msg[m + __popc(ball & ((1u << lane) - 1u))] = static_cast<int>(dg);
          m += __popc(ball);
        }
      }
      if (__any_sync(kFull, bad)) {
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
      zc = cd_row(ws, w, zc, ws.msg, m + mc + 1, j, CdX{xs, ws.cx, j, a.lut_col}, As, Ad, dst, prep, lane);
    }
    for (int i = rows + lane; i < MI; i += 32) {
      a.impact_node[k * MI + i] = -1;
      if (kMove && a.impact_kind) a.impact_kind[k * MI + i] = 0;
    }
    for (int i = rows * QOT_OUT + lane; i < MI * QOT_OUT; i += 32) a.impact_out[k * MI * QOT_OUT + i] = nan;
    if (lane == 0) {
      a.status[k] = st;
      a.n_impact[k] = cnt;
    }
  }
  if (zc) cd_flush(w, zc, prep, lane);
}

static int cfg_check(const qot_lp_graph_cfg_t* cfg, const char* who) {
  QOT_REQUIRE(cfg, "%s: null cfg", who);
  QOT_REQUIRE(cfg->F > 0 && cfg->L > 0 && cfg->Q > 0 && cfg->L <= 65535 && cfg->Q <= 65535 &&
                  static_cast<int64_t>(cfg->L) * cfg->Q < (1ll << 30), "%s: bad tensor extents", who);
  QOT_REQUIRE(cfg->i_conn >= 0 && cfg->i_conn < cfg->F, "%s: conn_id row out of range", who);
  return QOT_OK;
}

// shared by both entry points: argument checks, the once-per-device shared-memory opt-in, the launch
template <bool kMove>
static int cd_launch(const char* who, const qot_lp_graph_cfg_t* cfg, int64_t S, const double* freqs, const float* x,
                     const int64_t* node_ptr, const int64_t* rowptr, const int64_t* edge_index, int64_t N, int64_t E,
                     const int32_t* chan_node, int64_t K, const int64_t* node, const int64_t* sample,
                     const int64_t* link_ptr, const int32_t* links, int64_t n_links, const int32_t* q0,
                     const int32_t* width, const float* feat, const float* prepared, int32_t is_lut_index,
                     int32_t max_impact, float* out, int32_t* status, int32_t* n_impact, int64_t* impact_node,
                     int8_t* impact_kind, float* impact_out, cudaStream_t stream) {
  if (int rc = cfg_check(cfg, who)) return rc;
  QOT_REQUIRE(S >= 0 && N >= 0 && N < INT_MAX && E >= 0 && K >= 0 && n_links >= 0 && max_impact >= 0,
              "%s: bad size", who);
  QOT_REQUIRE(prepared && (reinterpret_cast<uintptr_t>(prepared) & 15) == 0, "%s: prepared must be 16-byte aligned",
              who);
  QOT_REQUIRE(is_lut_index >= 0 && is_lut_index < kF, "%s: is_lut_index out of range", who);
  if (K == 0) return QOT_OK;
  QOT_REQUIRE(sample && link_ptr && q0 && width && feat && out && status && n_impact && (n_links == 0 || links) &&
                  (max_impact == 0 || (impact_node && impact_out)) && (!kMove || node),
              "%s: null candidate or output array", who);
  QOT_REQUIRE(S == 0 || (freqs && x && node_ptr && rowptr && chan_node && (E == 0 || edge_index)),
              "%s: null state array", who);
  static std::atomic<unsigned long long> done{0};
  constexpr int smem = static_cast<int>(sizeof(CdSmem));
  if (int rc = once_per_device(done, [] {
        QOT_CUDA(cudaFuncSetAttribute(lp_candidate_kernel<kMove>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        return static_cast<int>(QOT_OK);
      }))
    return rc;
  CdArgs a;
  a.cfg = *cfg;
  a.S = S; a.N = N; a.E = E; a.K = K; a.n_links = n_links;
  a.freqs = freqs; a.x = x; a.node_ptr = node_ptr; a.rowptr = rowptr;
  a.edst = edge_index ? edge_index + E : nullptr;
  a.chan_node = chan_node;
  a.node = node;
  a.sample = sample; a.link_ptr = link_ptr; a.links = links; a.q0 = q0; a.width = width; a.feat = feat;
  a.prep = prepared; a.lut_col = is_lut_index; a.max_impact = max_impact;
  a.out = out; a.status = status; a.n_impact = n_impact; a.impact_node = impact_node;
  a.impact_kind = max_impact ? impact_kind : nullptr; a.impact_out = impact_out;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, cdiv(K, kCdWarps)));
  lp_candidate_kernel<kMove><<<grid, kCdThreads, smem, stream>>>(a);
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

extern "C" int qot_lightpath_candidates(const qot_lp_graph_cfg_t* cfg, int64_t S, const double* freqs,
                                        const float* x, const int64_t* node_ptr, const int64_t* rowptr,
                                        const int64_t* edge_index, int64_t N, int64_t E, const int32_t* chan_node,
                                        int64_t K, const int64_t* sample, const int64_t* link_ptr,
                                        const int32_t* links, int64_t n_links, const int32_t* q0,
                                        const int32_t* width, const float* feat, const float* prepared,
                                        int32_t is_lut_index, int32_t max_impact, float* out, int32_t* status,
                                        int32_t* n_impact, int64_t* impact_node, float* impact_out,
                                        void* stream_) {
  return cd_launch<false>("qot_lightpath_candidates", cfg, S, freqs, x, node_ptr, rowptr, edge_index, N, E, chan_node,
                          K, nullptr, sample, link_ptr, links, n_links, q0, width, feat, prepared, is_lut_index,
                          max_impact, out, status, n_impact, impact_node, nullptr, impact_out,
                          static_cast<cudaStream_t>(stream_));
}

extern "C" int qot_lightpath_reconfigure(const qot_lp_graph_cfg_t* cfg, int64_t S, const double* freqs,
                                         const float* x, const int64_t* node_ptr, const int64_t* rowptr,
                                         const int64_t* edge_index, int64_t N, int64_t E, const int32_t* chan_node,
                                         int64_t K, const int64_t* node, const int64_t* sample,
                                         const int64_t* link_ptr, const int32_t* links, int64_t n_links,
                                         const int32_t* q0, const int32_t* width, const float* feat,
                                         const float* prepared, int32_t is_lut_index, int32_t max_impact, float* out,
                                         int32_t* status, int32_t* n_impact, int64_t* impact_node,
                                         int8_t* impact_kind, float* impact_out, void* stream_) {
  return cd_launch<true>("qot_lightpath_reconfigure", cfg, S, freqs, x, node_ptr, rowptr, edge_index, N, E,
                         chan_node, K, node, sample, link_ptr, links, n_links, q0, width, feat, prepared,
                         is_lut_index, max_impact, out, status, n_impact, impact_node, impact_kind, impact_out,
                         static_cast<cudaStream_t>(stream_));
}
