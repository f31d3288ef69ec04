// LightpathGNN eval-mode forward as ONE persistent, warp-specialised, multi-stage kernel over MANY
// batches (lightpath_training/models.py:26-45 under model.eval(), as driven by
// lightpath_training/test.py:77-94; PyG semantics per SURVEY.md Appendix A.3 / A.5):
//
//   work item = a TILE of 16 consecutive graphs of one batch; a launch covers every tile of an array
//   of batch descriptors (reference layout: fp32 x, int64 edge_index, ptr / edge_ptr / lut_ptr);
//   one CTA per SM loops over tiles  bid, bid + grid, bid + 2*grid, ...
//
//   warp 0            PRODUCER.  Its 32 lanes look 32 tiles ahead (tile extents = 4 index loads each, all in
//                     flight at once), then per tile: wait for a free stage, 51 x 8-byte cp.async for the
//                     tile's ptr / edge_ptr / lut_ptr rows, and ONE elected lane issues two cp.async.bulk
//                     copies -- the x window (20 B/node) and the window of the DESTINATION row of
//                     edge_index (8 B/edge) -- completing on the stage's `full` mbarrier.
//   warps 1..12       three CONSUMER groups of four warps.  Group q takes the CTA's tiles k = q (mod 3):
//                     8 lanes per graph -- LUT flag scan, destination scan (contiguous runs, one compare
//                     per slot), the few sources of the LUT row fetched from the source row in global
//                     memory, 4-head attention softmax over 5-float messages (z = sum_j alpha_ij x_j),
//                     then the z row (20 floats) goes to the readout head.  The stage is released on its
//                     `empty` mbarrier as soon as the slabs are dead.
//   (head)            see lp_head_kernel below / the tcgen05 head warps.
//
// Nothing is re-read: the parameter block, the attention vectors and the barrier setup are loaded once
// per CTA, tile extents once per 32 tiles, and every compulsory byte of a graph is requested by one
// asynchronous copy several tiles before it is needed, so the three dependent DRAM round trips of the
// one-launch-per-batch kernel (extents -> slabs -> sources) overlap across tiles instead of
// serialising inside a CTA.  Deterministic: edges of a row are consumed in edge order, fixed trees.
#include <algorithm>
#include <type_traits>

#include "lightpath_common.cuh"

namespace qot {

constexpr int kTG = 16;                    // graphs per tile
constexpr int kTNodes = 704;               // x window: mean 512 nodes + 3.4 sigma (sigma = 4 * 14.1)
constexpr int kTEdges = 2688;              // destination window: mean 1984 edges + 3.1 sigma
constexpr int kTMaxE = 248;                // per graph: 8 lanes x 31 contiguous edges (bit mask per lane)
// Two builds of the kernel.  kHead = false: consumers write z rows to the batch's workspace and lp_stream_head_kernel
// finishes them (one more launch).  kHead = true (default): the readout head runs INSIDE the kernel on the 5th-generation
// tensor cores -- four epilogue warps + one MMA-issuing warp per CTA, accumulators in TMEM (see st_head_epilogue).
#ifndef QOT_ST_WARPS
#define QOT_ST_WARPS 15
#endif
#ifndef QOT_ST_XSTAGES
#define QOT_ST_XSTAGES 7
#endif
#ifndef QOT_ST_DSTAGES
#define QOT_ST_DSTAGES 4
#endif
#ifndef QOT_STH_WARPS
#define QOT_STH_WARPS 14
#endif
#ifndef QOT_STH_XSTAGES
#define QOT_STH_XSTAGES 6
#endif
#ifndef QOT_STH_DSTAGES
#define QOT_STH_DSTAGES 3
#endif
template <bool kHead> struct StCfg;
template <> struct StCfg<false> {
  static constexpr int kX = QOT_ST_XSTAGES;      // x ring: a stage lives until its tile's attention rows are out
  static constexpr int kD = QOT_ST_DSTAGES;      // destination ring: a stage is dead as soon as the tile has been scanned
  static constexpr int kConsumers = QOT_ST_WARPS;
  static constexpr int kThreads = 32 * (1 + kConsumers);          // warp 0 producer, the rest consumers
};
template <> struct StCfg<true> {
  static constexpr int kX = QOT_STH_XSTAGES;
  static constexpr int kD = QOT_STH_DSTAGES;
  static constexpr int kConsumers = QOT_STH_WARPS;
  // warp 0 producer, 1 MMA issuer, 2-3 consumers, 4-7 epilogue (TMEM lane quarter = warp - 4), 8.. consumers
  static constexpr int kThreads = 32 * (8 + kConsumers - 2);
};
constexpr int kStGroupWarps = 4;           // a tile = 4 quarter-tiles of 4 graphs; a consumer warp takes one at a time
constexpr int kStXBytes = kTNodes * kF * 4;
constexpr int kStDBytes = kTEdges * 8;

struct alignas(16) StTileInfo {
  qot_lp_batch_t d;                        // the batch descriptor, copied asynchronously with the index rows
  int64_t g0;                              // first graph of the tile (index inside its batch)
  int64_t nb0, eb0;                        // first node / edge staged
  int xn, en;                              // nodes / edges staged (0: window unusable, graphs take the generic path)
  unsigned xlead, dlead;                   // bytes between the 16-byte aligned copy start and the first element
  int ng;                                  // graphs in the tile
  int pad;
};
static_assert(sizeof(qot_lp_batch_t) == 128, "the descriptor is copied as eight 16-byte pieces");

struct alignas(128) StStage {
  alignas(128) unsigned char xs[kStXBytes + 16];
  alignas(16) long long ptrs[3][kTG + 2];  // ptr / edge_ptr / lut_ptr rows of the tile (kTG + 1 entries each)
  StTileInfo info;
};
struct alignas(128) StDStage {
  alignas(128) unsigned char ds[kStDBytes + 16];
};

struct StGenericArgs {                     // tile fields the generic path needs after the stage is handed back
  const float* x;
  const int64_t* esrc;
  const int64_t* edst;
  float* z;
  float* out;
  int64_t* lut_batch;
  int32_t* lut_node;
  int32_t* status;
  int64_t N, E, g0;
  int64_t p[4][6];                         // per graph of the warp: n0 n1 e0 e1 l0 l1
};

struct StWarpScratch {                     // per consumer warp
  StGenericArgs gargs;
  int msg[4][kSubMsg];
  int raw[4][kSubMsg];                     // kSym: the LUT node's out-run before ranking
};

constexpr int kZPitch = 21;                // floats per staged z row (odd: the epilogue's row-per-lane reads hit 32 banks)
constexpr int kGroupTiles = 8;             // tiles per readout group: 8 x 16 graphs = the 128 rows of one MMA
// shared memory of the in-kernel readout head
struct StHeadSmem {
  alignas(1024) float b2[2][4][32 * 32];   // mlp.0 weight, tcgen05 B operand: [hi | lo][k-block][row n][32 floats], swizzled
  float zrow[2][128 * kZPitch];            // z rows of a group (double buffered), row = (tile % 8) * 16 + graph slot
  float* optr[2][128];                     // where the row's 3 outputs go; nullptr: the slot holds no row
  alignas(8) unsigned long long zfull[2];  // 32 quarter-tile arrivals: the group's rows are staged
  alignas(8) unsigned long long zfree[2];  // 4 epilogue warps: the buffer has been read
  alignas(8) unsigned long long aready;    // 4 epilogue warps: the A operand (hidden activations) is in TMEM
  alignas(8) unsigned long long dready;    // tcgen05.commit: the accumulator is complete
  unsigned tmem_base;
  // readout-head parameters read by every epilogue thread (broadcast): with ~225 KB of the SM's 256 KB configured as
  // shared memory almost no L1 is left, so nothing on a hot path may depend on cached global loads
  alignas(16) float wf[kHC * kF];          // [h][f][32]: folded GAT projection (BN scale inside)
  alignas(16) float shift[kHC];
  alignas(16) float b1[kHid];
  alignas(16) float w2[QOT_OUT * kHid];
  float bo[4];
};
struct StNoHead {};

template <bool kHead>
struct StSmemT {
  typename std::conditional<kHead, StHeadSmem, StNoHead>::type head;   // first: 1024-byte aligned operand tiles
  StDStage dstage[StCfg<kHead>::kD];       // before the x ring: the scan's masked over-reads past a window stay inside the block
  StStage stage[StCfg<kHead>::kX];
  float4 asp[8][6];                        // attention source vectors per lane slot (lp_prepare_kernel's kOffAsP table)
  float4 adp[4][kF];                       // attention destination vectors per head-slot group (kOffAdP table)
  StWarpScratch wsc[StCfg<kHead>::kConsumers];
  float gen[256];                          // generic path scratch (one graph at a time per CTA, under gen_lock)
  alignas(8) unsigned long long full[StCfg<kHead>::kX];    // x window + destination window + index rows of a tile landed
  alignas(8) unsigned long long empty[StCfg<kHead>::kX];   // x stage released (4 quarter-tiles)
  alignas(8) unsigned long long dempty[StCfg<kHead>::kD];  // destination stage released (4 quarter-tiles)
  int next_unit;                           // quarter-tiles handed out so far (consumer warps claim them in order)
  int gen_lock;
};
// Every function reaches the block's shared memory through this accessor (not through a reference parameter): the
// address then provably lies in the shared window and the compiler emits LDS / STS / ATOMS instead of generic
// LD / ST / ATOM, which cost an address-space check and the long-scoreboard path on every access.
extern __shared__ __align__(1024) char st_smem_raw[];
template <bool kHead>
__device__ __forceinline__ StSmemT<kHead>& st_smem() {
  const unsigned off = (1024u - (static_cast<unsigned>(__cvta_generic_to_shared(st_smem_raw)) & 1023u)) & 1023u;
  return *reinterpret_cast<StSmemT<kHead>*>(st_smem_raw + off);
}
static_assert(sizeof(StSmemT<false>) + 1024 <= 227 * 1024, "lp_stream_kernel: shared memory over the 227 KB block limit");
static_assert(sizeof(StSmemT<true>) + 1024 <= 227 * 1024, "lp_stream_kernel<head>: shared memory over the 227 KB block limit");

#ifdef QOT_ST_TRACE
// debug build only (scripts/build_variant.sh ... -DQOT_ST_TRACE): per-CTA cycle sums, 8 slots per CTA:
// 0 producer wait-empty, 1 producer issue, 2 consumer wait-full (all warps), 3 consumer work (incl. 4), 4 consumer wait for
// a free z buffer, 5 epilogue wait for a staged group, 6 epilogue wait for the MMAs, 7 epilogue total
__device__ unsigned long long* g_st_trace = nullptr;
#define ST_DECL() long long st_acc_[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define ST_T0() const long long st_t0_ = clock64()
#define ST_T1() const long long st_t1_ = clock64()
#define ST_PARAM , long long* st_acc_
#define ST_ARG , st_acc_
#define ST_ACC1(slot) do { st_acc_[slot] += clock64() - st_t1_; } while (0)
#define ST_ACC(slot) do { st_acc_[slot] += clock64() - st_t0_; } while (0)
#define ST_FLUSH() do { if (g_st_trace && lane == 0) for (int i_ = 0; i_ < 8; ++i_) if (st_acc_[i_]) atomicAdd(g_st_trace + blockIdx.x * 8 + i_, static_cast<unsigned long long>(st_acc_[i_])); } while (0)
#else
#define ST_DECL() do {} while (0)
#define ST_T0() do {} while (0)
#define ST_T1() do {} while (0)
#define ST_PARAM
#define ST_ARG
#define ST_ACC1(slot) do {} while (0)
#define ST_ACC(slot) do {} while (0)
#define ST_FLUSH() do {} while (0)
#endif
__device__ __forceinline__ unsigned st_smem_u32(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
// try_wait with an explicit suspend-time hint: a waiting warp sleeps in hardware until the phase completes (or the
// hint expires) instead of re-issuing the poll -- 57 % of all issued instructions were polls without it, and they
// compete with the producer warp for issue slots
#ifndef QOT_ST_SUSPEND_NS
#define QOT_ST_SUSPEND_NS 20000
#endif
__device__ __forceinline__ bool st_try_wait(unsigned bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3; selp.u32 %0, 1, 0, p; }"
      : "=r"(ok) : "r"(bar), "r"(parity), "r"(QOT_ST_SUSPEND_NS) : "memory");
  return ok != 0u;
}
// bounded wait: a wedged barrier ends the kernel after ~2 s of wall clock (status bit 2), it never hangs the GPU.
// Between polls the warp sleeps `kSleepNs` (ncu: without it 13 % of all issued instructions were polls of warps with
// nothing to do -- the suspend-time hint alone does not park them -- taking issue slots from the working warps).
template <unsigned kSleepNs = 40>
__device__ __forceinline__ bool st_wait(unsigned bar, unsigned parity) {
  if (st_try_wait(bar, parity)) return true;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (;;) {
#pragma unroll 1
    for (int i = 0; i < 256; ++i) {
      __nanosleep(kSleepNs);
      if (st_try_wait(bar, parity)) return true;
    }
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    if (t1 - t0 > 2000000000ull) return false;
  }
}
__device__ __forceinline__ void st_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void st_mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(st_smem_u32(bar)), "r"(count) : "memory");
}

// ------------------------------------------------------------------------------------------------
// producer: one warp
// ------------------------------------------------------------------------------------------------
template <bool kHead>
__device__ __noinline__ void st_producer(const qot_lp_batch_t* __restrict__ bt, int nb, int64_t tpb,
                                         int64_t tile_base, int64_t total_tiles, int lane) {
  StSmemT<kHead>& sm = st_smem<kHead>();
  const int64_t G = gridDim.x;
  const int64_t my_tiles = (total_tiles - blockIdx.x + G - 1) / G;
  ST_DECL();
  for (int64_t kb = 0; kb < my_tiles; kb += 32) {
    // ---- look-ahead: lane j owns tile kb + j of this CTA and fetches EVERYTHING its issue needs from global memory
    // (descriptor fields, tile extents) -- 32 tiles' worth of dependent loads in flight at once, so the per-tile
    // issue path below touches registers and shared memory only
    int b = 0;
    long long g0 = 0, nb0 = 0, nb1 = 0, eb0 = 0, eb1 = 0, dN = 0, dE = 0, dB = 0;
    const float* dx = nullptr;
    const int64_t *dei = nullptr, *dptr = nullptr, *deptr = nullptr, *dlptr = nullptr;
    if (kb + lane < my_tiles) {
      const int64_t T = tile_base + blockIdx.x + (kb + lane) * G;
      b = st_batch_of(bt, nb, tpb, tile_base, T);
      const qot_lp_batch_t& d = bt[b];
      dx = d.x; dei = d.edge_index; dptr = d.ptr; deptr = d.edge_ptr; dlptr = d.lut_ptr;
      dN = d.N; dE = d.E; dB = d.B;
      g0 = (T - d.tile0) * kTG;
      const int64_t gE = min(static_cast<int64_t>(g0 + kTG), static_cast<int64_t>(dB));
      nb0 = dptr[g0]; nb1 = dptr[gE];
      eb0 = deptr[g0]; eb1 = deptr[gE];
    }
    const int cnt = static_cast<int>(min(static_cast<int64_t>(32), my_tiles - kb));
    for (int j = 0; j < cnt; ++j) {
      const int64_t k = kb + j;
      constexpr int kStStages = StCfg<kHead>::kX, kStDStages = StCfg<kHead>::kD;
      const int s = static_cast<int>(k % kStStages);
      const unsigned ph = static_cast<unsigned>((k / kStStages) & 1);
      StStage& st = sm.stage[s];
      const int sd_ = static_cast<int>(k % kStDStages);
      StDStage& dst_stage = sm.dstage[sd_];
      const unsigned fbar = st_smem_u32(&sm.full[s]);
      {
        ST_T0();
        st_wait(st_smem_u32(&sm.empty[s]), ph ^ 1u);     // consumers released the stages' previous tiles
        st_wait(st_smem_u32(&sm.dempty[sd_]), static_cast<unsigned>((k / kStDStages) & 1) ^ 1u);
        ST_ACC(0);
      }
      ST_T0();
      const int tb = __shfl_sync(kFull, b, j);
      const long long tg0 = __shfl_sync(kFull, g0, j), tB = __shfl_sync(kFull, dB, j);
      const int64_t* tptr = reinterpret_cast<const int64_t*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(dptr), j));
      const int64_t* teptr = reinterpret_cast<const int64_t*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(deptr), j));
      const int64_t* tlptr = reinterpret_cast<const int64_t*>(__shfl_sync(kFull, reinterpret_cast<unsigned long long>(dlptr), j));
      // ---- the tile's index rows (3 x (kTG + 1) entries, 8-byte pieces) and its batch descriptor (8 x 16 bytes),
      // all asynchronous: they arrive on the stage's `full` barrier like the two windows
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int idx = lane + 32 * r;
        if (idx < 3 * (kTG + 1)) {
          const int which = idx / (kTG + 1), i = idx % (kTG + 1);
          const int64_t gi = min(static_cast<int64_t>(tg0 + i), static_cast<int64_t>(tB));
          const int64_t* src = (which == 0 ? tptr : which == 1 ? teptr : tlptr) + gi;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(st_smem_u32(&st.ptrs[which][i])), "l"(src) : "memory");
        }
      }
      if (lane >= 24)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                     ::"r"(st_smem_u32(reinterpret_cast<char*>(&st.info.d) + 16 * (lane - 24))),
                       "l"(reinterpret_cast<const char*>(bt + tb) + 16 * (lane - 24)) : "memory");
      asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(fbar) : "memory");
      // lane j still holds the tile's remaining values: it sizes the windows and issues the bulk copies itself
      if (lane == j) {
        // ---- windows: nodes [nb0, nb0 + xn), edges [eb0, eb0 + en), copied from 16-byte aligned addresses;
        // a window that does not fit (or nonsense offsets) is not staged: its graphs take the generic path
        int xn = 0, en = 0;
        if (nb0 >= 0 && nb1 >= nb0 && nb1 <= dN && nb1 - nb0 <= kTNodes) xn = static_cast<int>(nb1 - nb0);
        if (eb0 >= 0 && eb1 >= eb0 && eb1 <= dE && eb1 - eb0 <= kTEdges) en = static_cast<int>(eb1 - eb0);
        if (xn == 0 || (en == 0 && eb1 != eb0)) { xn = 0; en = 0; }
        const int64_t* edst = dei + dE;
        const uintptr_t xa = reinterpret_cast<uintptr_t>(dx) + static_cast<uintptr_t>(xn > 0 ? nb0 : 0) * (kF * 4);
        const uintptr_t da = reinterpret_cast<uintptr_t>(edst) + static_cast<uintptr_t>(en > 0 ? eb0 : 0) * 8;
        const unsigned xlead = static_cast<unsigned>(xa & 15), dlead = static_cast<unsigned>(da & 15);
        const uintptr_t xs0 = xa - xlead, ds0 = da - dlead;
        const unsigned xspan = xlead + static_cast<unsigned>(xn) * (kF * 4), dspan = dlead + static_cast<unsigned>(en) * 8;
        unsigned xbytes = (xspan + 15u) & ~15u, dbytes = (dspan + 15u) & ~15u;
        // never read past the end of a tensor: the few bytes a rounded-up window would add are copied by hand
        if (xs0 + xbytes > reinterpret_cast<uintptr_t>(dx) + static_cast<uintptr_t>(dN) * (kF * 4)) xbytes = xspan & ~15u;
        if (ds0 + dbytes > reinterpret_cast<uintptr_t>(edst) + static_cast<uintptr_t>(dE) * 8) dbytes = dspan & ~15u;
        if (xn == 0) xbytes = 0;
        if (en == 0) dbytes = 0;
        if (xn > 0)
          for (unsigned o = xbytes; o < xspan; o += 4)
            *reinterpret_cast<float*>(st.xs + o) = *reinterpret_cast<const float*>(xs0 + o);
        if (en > 0 && dspan > dbytes)
          *reinterpret_cast<long long*>(dst_stage.ds + dbytes) = *reinterpret_cast<const long long*>(ds0 + dbytes);
        StTileInfo& ti = st.info;
        ti.g0 = g0; ti.nb0 = nb0; ti.eb0 = eb0;
        ti.xn = xn; ti.en = en; ti.xlead = xlead; ti.dlead = dlead;
        ti.ng = static_cast<int>(min(static_cast<int64_t>(kTG), static_cast<int64_t>(dB - g0)));
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fbar), "r"(xbytes + dbytes) : "memory");
        if (xbytes)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(st_smem_u32(st.xs)), "l"(xs0), "r"(xbytes), "r"(fbar) : "memory");
        if (dbytes)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                       ::"r"(st_smem_u32(dst_stage.ds)), "l"(ds0), "r"(dbytes), "r"(fbar) : "memory");
      }
      __syncwarp();
      ST_ACC(1);
    }
  }
  ST_FLUSH();
}

// generic path: graphs of this warp the fast path declined (over the caps, several / no LUT rows, hub rows,
// foreign ids): one warp per graph, straight from global memory.  kHead: the FP32 readout head of the row runs here
// too and writes `out`; otherwise the z row goes to the batch's workspace for lp_stream_head_kernel.  The scratch is
// one per CTA (these graphs are rare), taken under a lock.
template <bool kHead>
__device__ __noinline__ void st_generic(int cw, unsigned todo, const float* __restrict__ prep, int lut_col, int lane) {
  StSmemT<kHead>& sm = st_smem<kHead>();
  const StGenericArgs& ga = sm.wsc[cw].gargs;
  float* scratch = sm.gen;
  int* lock = &sm.gen_lock;
  const float* gx = ga.x;
  const int64_t N = ga.N;
  if (lane == 0)
    while (atomicCAS(lock, 0, 1) != 0) __nanosleep(200);
  __syncwarp();
  float* s_y = scratch;                    // 128 floats (kHead)
  float* s_z = scratch + 128;              // 32
  int* s_m = reinterpret_cast<int*>(scratch + 160);   // 64
#pragma unroll 1
  for (int s = 0; s < 4; ++s) {
    if (!((todo >> s) & 1u)) continue;
    const int64_t gn0 = ga.p[s][0], gn1 = ga.p[s][1], ge0 = ga.p[s][2], ge1 = ga.p[s][3], gl0 = ga.p[s][4], gl1 = ga.p[s][5];
    int64_t orow = gl0;
    int found = 0;
    if (gn0 >= 0 && gn1 <= N && ge0 >= 0 && ge1 <= ga.E) {
      for (int64_t nbq = gn0; nbq < gn1; nbq += 32) {
        const int64_t node = nbq + lane;
        unsigned mask = __ballot_sync(kFull, node < gn1 && gx[node * kF + lut_col] == 1.0f);
        while (mask) {
          const int bit = __ffs(mask) - 1;
          mask &= mask - 1;
          ++found;
          if (orow < gl1) {                                      // never write past this graph's rows
            const int64_t i = nbq + bit;
            if constexpr (kHead) {
              const float ov = lut_row_global<true>(XRaw{gx}, ga.esrc, ga.edst, ge0, ge1, N, i, prep, prep + kOffWf, s_m, s_z, s_y, lane);
              if (lane < QOT_OUT) ga.out[orow * QOT_OUT + lane] = ov;
            } else {
              lut_row_global<false>(XRaw{gx}, ga.esrc, ga.edst, ge0, ge1, N, i, prep, nullptr, s_m, s_z, nullptr, lane);
              if (lane < kHeads * kF) ga.z[orow * (kHeads * kF) + lane] = s_z[(lane / kF) * 8 + lane % kF];
            }
            if (lane == 0) {
              ga.lut_batch[orow] = ga.g0 + s;
              ga.lut_node[orow] = static_cast<int32_t>(i);
            }
            __syncwarp();
            ++orow;
          }
        }
      }
    }
    if (lane == 0 && found != gl1 - gl0) atomicOr(ga.status, 1);
  }
  __syncwarp();
  if (lane == 0) {
    __threadfence_block();
    atomicExch(lock, 0);
  }
}

// One tile.  Everything per graph is kept as 32-bit offsets inside the tile's windows (the 64-bit index rows stay in
// the stage and are re-read where a global index is needed): registers are what bounds the consumer-warp count.
template <bool kHead, bool kSym>
__device__ __forceinline__ void st_consume_tile(int k, int cw, const float* __restrict__ prep, int lut_col, int gw,
                                                int lane ST_PARAM) {
  StSmemT<kHead>& sm = st_smem<kHead>();
  StWarpScratch& gs = sm.wsc[cw];
  StStage& st = sm.stage[k % StCfg<kHead>::kX];
  const StDStage& dstg = sm.dstage[k % StCfg<kHead>::kD];
  const unsigned ebar = st_smem_u32(&sm.empty[k % StCfg<kHead>::kX]), dbar = st_smem_u32(&sm.dempty[k % StCfg<kHead>::kD]);
  const float4 (*__restrict__ asp)[6] = sm.asp;
  const int sg = lane >> 3, sl = lane & 7;
  const int gl = gw * 4 + sg;                          // graph slot inside the tile
  const StTileInfo& ti = st.info;
  int n = 0, ne = 0, xoff = 0, eoff = 0, lrows = 0;
  bool active, fits;
  {
    const int64_t n0 = st.ptrs[0][gl], n1 = st.ptrs[0][gl + 1];
    const int64_t e0 = st.ptrs[1][gl], e1 = st.ptrs[1][gl + 1];
    const int64_t l0 = st.ptrs[2][gl], l1 = st.ptrs[2][gl + 1];
    const int64_t nb0 = ti.nb0, eb0 = ti.eb0;
    const int xn = ti.xn, en = ti.en;
    active = gl < ti.ng;
    fits = active && xn > 0 && n1 >= n0 && e1 >= e0 && (n1 - n0) <= kMaxN && (e1 - e0) <= kTMaxE &&
           n0 >= nb0 && (n1 - nb0) <= xn && e0 >= eb0 && (e1 - eb0) <= en && l1 >= l0 && (l1 - l0) <= kMaxN;
    if (fits) {
      n = static_cast<int>(n1 - n0); ne = static_cast<int>(e1 - e0);
      xoff = static_cast<int>(n0 - nb0); eoff = static_cast<int>(e0 - eb0);
      lrows = static_cast<int>(l1 - l0);
    }
    if (active && ti.g0 + gl == ti.d.B - 1 && sl == 0) ti.d.n_lut[0] = static_cast<int32_t>(l1);
  }
  const float* sx = reinterpret_cast<const float*>(st.xs + ti.xlead) + xoff * kF;
  const long long* sd = reinterpret_cast<const long long*>(dstg.ds + ti.dlead) + eoff;
  const int hx = sl >> 1;
  const bool odd = (sl & 1) != 0;

  // ---- LUT node(s) of the graph: a per-lane bit per node, then one count and one minimum over the 8 lanes
  int cnt = 0, il = -1;
  {
    unsigned m = 0u;
    const int rmax = (__reduce_max_sync(kFull, n) + 7) >> 3;
#pragma unroll
    for (int r = 0; r < kMaxN / 8; ++r) {
      if (r < rmax) {
        const int node = sl + 8 * r;
        if (node < n && sx[node * kF + lut_col] == 1.0f) m |= 1u << r;
      }
    }
    cnt = __popc(m);
    int first = m ? 8 * (__ffs(m) - 1) + sl : 0x7fff;
#pragma unroll
    for (int o = 1; o <= 4; o <<= 1) {
      cnt += __shfl_xor_sync(kFull, cnt, o);
      first = min(first, __shfl_xor_sync(kFull, first, o));
    }
    if (cnt) il = first;
  }
  bool ok = fits && cnt == 1 && lrows == 1;            // fast row: exactly one LUT node, as lut_ptr says
  if (fits && sl == 0 && cnt != lrows) atomicOr(ti.d.status, 1);   // lut_ptr does not describe this x

  int* msg = gs.msg[sg];
  int mc = 0;
  if constexpr (kSym) {
    // ---- layout invariant verified by the store (PackedGraphStore.verify_layout): every graph is symmetric, without
    // duplicate edges, its edges grouped by source ascending, every endpoint inside the graph (what from_networkx
    // emits for an undirected graph, SURVEY.md A.6).  Then indeg(u) = outdeg(u) for every node, the out-run of the
    // LUT node il starts at #{edges with dst < il}, is #{dst == il} long, and its destinations ARE the sources of
    // il's in-edges; in edge order those sources ascend.  So the scan only counts -- on the low words: verified ids
    // are < N < 2^31 -- and nothing is read from the source row.
    const int c = ((ne + 7) >> 3) | 1;                 // odd run length: the 8 lanes' reads hit distinct banks
    const int eb = sl * c;
    const int tmax = ok ? min(c, ne - eb) : 0;
    const int cmax = __reduce_max_sync(kFull, tmax);
    const int target = static_cast<int>(st.ptrs[0][gl]) + il;
    const int* sde = reinterpret_cast<const int*>(sd + eb);
    // four independent accumulator pairs (slot mod 4): the predicated ORs of consecutive slots do not chain
    unsigned em[4] = {0u, 0u, 0u, 0u}, lm[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int t4 = 0; t4 < 32; t4 += 4) {
      if (t4 < cmax) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int t = t4 + i;
          if (t < 31) {
            const int d = sde[2 * t];                  // masked below: slots past the run stay inside the block's memory
            asm("{ .reg .pred p, q;\n\t"
                "setp.eq.s32 p, %2, %3;\n\t"
                "setp.lt.s32 q, %2, %3;\n\t"
                "@p or.b32 %0, %0, %4;\n\t"
                "@q or.b32 %1, %1, %4; }"
                : "+r"(em[i]), "+r"(lm[i]) : "r"(d), "r"(target), "r"(1u << t));
          }
        }
      }
    }
    const unsigned vm = (1u << max(tmax, 0)) - 1u;     // tmax <= 31
    int pack = __popc((em[0] | em[1] | em[2] | em[3]) & vm) | (__popc((lm[0] | lm[1] | lm[2] | lm[3]) & vm) << 16);
#pragma unroll
    for (int o = 1; o <= 4; o <<= 1) pack += __shfl_xor_sync(kFull, pack, o);
    const int deg = pack & 0xffff, start = pack >> 16;
    if (deg > kSubMsg - 1) ok = false;                 // hub row: generic path
    // the out-run of il: <= 15 destinations, two per lane; self loops dropped, ascending order by ranking
    int* raw = gs.raw[sg];
    int v0 = 0x7fffffff, v1 = 0x7fffffff;
    bool bad = false;
    if (ok) {
      const int n0i = target - il;
      if (sl < deg) {
        const int w = static_cast<int>(sd[start + sl]) - n0i;
        bad |= w < 0 || w >= n;
        if (w != il) v0 = w;
      }
      if (sl + 8 < deg) {
        const int w = static_cast<int>(sd[start + sl + 8]) - n0i;
        bad |= w < 0 || w >= n;
        if (w != il) v1 = w;
      }
    }
    raw[sl] = v0;
    raw[sl + 8] = v1;
    if (((__ballot_sync(kFull, bad) >> (8 * sg)) & 0xffu) != 0u) ok = false;   // not a node of this graph: generic path
    const int dmax = __reduce_max_sync(kFull, ok ? deg : 0);
    __syncwarp();
    if (lane == 0) st_arrive(dbar);                    // last read of the destination window: its stage may be refilled
    int r0 = 0, r1 = 0;
    for (int j = 0; j < dmax; ++j) {
      const int w = raw[j];                             // entries past deg hold INT_MAX: they rank nobody down
      r0 += w < v0;
      r1 += w < v1;
    }
    const bool k0 = ok && v0 != 0x7fffffff, k1 = ok && v1 != 0x7fffffff;
    if (k0) msg[r0] = v0;
    if (k1) msg[r1] = v1;
    const unsigned kb0 = (__ballot_sync(kFull, k0) >> (8 * sg)) & 0xffu, kb1 = (__ballot_sync(kFull, k1) >> (8 * sg)) & 0xffu;
    mc = __popc(kb0) + __popc(kb1);
  } else {
    // ---- in-edges of the LUT node: lane sl scans edges [sl*c, sl*c + c) of its graph (c odd: the 8-byte reads of
    // the 8 lanes fall into distinct banks); one predicate per slot
    {
      const int c = ((ne + 7) >> 3) | 1;
      const int eb = sl * c;
      const int tmax = ok ? min(c, ne - eb) : 0;
      const int cmax = __reduce_max_sync(kFull, tmax);
      const long long target = st.ptrs[0][gl] + il;
      const int tlo = static_cast<int>(target), thi = static_cast<int>(target >> 32);
      // unconditional 8-byte reads: slots past the lane's run stay inside the block's shared memory and are masked
      // by t < tmax
      const int2* sde = reinterpret_cast<const int2*>(sd + eb);
      unsigned hm = 0u;
#pragma unroll
      for (int t4 = 0; t4 < 32; t4 += 4) {
        if (t4 < cmax) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int t = t4 + i;
            if (t < 31) {
              const int2 d = sde[t];
              asm("{ .reg .pred p;\n\t"
                  "setp.eq.s32 p, %1, %3;\n\t"
                  "setp.eq.and.s32 p, %2, %4, p;\n\t"
                  "@p or.b32 %0, %0, %5; }"
                  : "+r"(hm) : "r"(d.x), "r"(d.y), "r"(tlo), "r"(thi), "r"(1u << t));
            }
          }
        }
      }
      hm &= (1u << max(tmax, 0)) - 1u;                   // tmax <= 31
      const int h = __popc(hm);
      int incl = h;
#pragma unroll
      for (int o = 1; o <= 4; o <<= 1) {
        const int up = __shfl_up_sync(kFull, incl, o, 8);
        if (sl >= o) incl += up;
      }
      mc = __shfl_sync(kFull, incl, (lane & ~7) + 7);
      int pos = incl - h;
      while (hm) {
        const int t = __ffs(hm) - 1;
        hm &= hm - 1u;
        if (pos < kSubMsg - 1) msg[pos] = eb + t;
        ++pos;
      }
    }
    if (mc > kSubMsg - 1) ok = false;                    // hub row: generic path
    __syncwarp();
    if (lane == 0) st_arrive(dbar);                      // last read of the destination window: its stage may be refilled
    // ---- sources of those edges (one gather per 8); self loops / out-of-range ids dropped, order kept
    {
      int kept = 0;
      bool outside = false;
      const int64_t* __restrict__ esrc = ti.d.edge_index + st.ptrs[1][gl];
      const int64_t n0 = st.ptrs[0][gl], N = ti.d.N;
#pragma unroll
      for (int t0 = 0; t0 < kSubMsg; t0 += 8) {
        if (__any_sync(kFull, ok && t0 < mc)) {
          const int t = t0 + sl;
          long long sj = -1;
          if (ok && t < mc) sj = esrc[msg[t]];
          const bool inN = static_cast<uint64_t>(sj) < static_cast<uint64_t>(N);
          const long long sloc = sj - n0;
          const bool inslab = sloc >= 0 && sloc < n;
          const bool keep = inslab && sloc != il;
          outside |= ((__ballot_sync(kFull, inN && !inslab) >> (8 * sg)) & 0xffu) != 0u;
          const unsigned sub = (__ballot_sync(kFull, keep) >> (8 * sg)) & 0xffu;
          __syncwarp();
          if (keep) msg[kept + __popc(sub & ((1u << sl) - 1u))] = static_cast<int>(sloc);
          kept += __popc(sub);
          __syncwarp();
        }
      }
      if (outside) ok = false;                           // a source outside the graph's node range: generic path
      mc = kept;
    }
  }
  if (ok && sl == 0) msg[mc] = il;                     // the appended self loop comes last
  ++mc;
  __syncwarp();

  // ---- attention: lane = message slot, all 4 heads per lane.  The 24 sums per graph (4 heads x (x0..x4, 1)) are
  // reduce-scattered: three exchange steps, each lane sends the half it does not keep -- statically the upper
  // half of its registers thanks to the slot permutation (tables built once by lp_prepare_kernel)
  {
    float d[kHeads];
    const int ils = ok ? il : 0;
#pragma unroll
    for (int i = 0; i < kHeads; ++i) d[i] = 0.f;
#pragma unroll
    for (int k = 0; k < kF; ++k) {
      const float xi = sx[ils * kF + k];
      const float4 b = sm.adp[hx][k];
      d[0] = fmaf(xi, b.x, d[0]); d[1] = fmaf(xi, b.y, d[1]);
      d[2] = fmaf(xi, b.z, d[2]); d[3] = fmaf(xi, b.w, d[3]);
    }
    float mx[kHeads], acc3[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < kHeads; ++i) mx[i] = -INFINITY;
    const int o0 = odd ? 3 : 0;
#pragma unroll
    for (int r0 = 0; r0 < kSubMsg; r0 += 8) {
      if (__any_sync(kFull, ok && r0 < mc)) {
        const bool valid = ok && r0 + sl < mc;
        const float* xr = sx + (valid ? msg[r0 + sl] : 0) * kF;
        float q[6];
        const float x2 = xr[2];
        q[0] = xr[o0]; q[1] = xr[o0 + 1]; q[3] = xr[3 - o0]; q[4] = xr[4 - o0];
        q[2] = odd ? 1.0f : x2;
        q[5] = odd ? x2 : 1.0f;
        float a[kHeads], mr[kHeads], m2[kHeads];
#pragma unroll
        for (int i = 0; i < kHeads; ++i) a[i] = d[i];
#pragma unroll
        for (int m = 0; m < 6; ++m) {                       // the ONE slot carries weight 0
          const float4 w = asp[sl][m];
          a[0] = fmaf(q[m], w.x, a[0]); a[1] = fmaf(q[m], w.y, a[1]);
          a[2] = fmaf(q[m], w.z, a[2]); a[3] = fmaf(q[m], w.w, a[3]);
        }
#pragma unroll
        for (int i = 0; i < kHeads; ++i) {
          const float t = a[i] > 0.f ? a[i] : 0.2f * a[i];
          a[i] = valid ? t : -INFINITY;
        }
#pragma unroll
        for (int i = 0; i < kHeads; ++i) mr[i] = fmaxf(a[i], __shfl_xor_sync(kFull, a[i], 1));
#pragma unroll
        for (int i = 0; i < kHeads; ++i) m2[i] = fmaxf(mr[i], __shfl_xor_sync(kFull, mr[i ^ 1], 2));
#pragma unroll
        for (int i = 0; i < kHeads; ++i) mr[i] = fmaxf(m2[i], __shfl_xor_sync(kFull, m2[i ^ 2], 4));
        float v[24];
        float scarg = 0.f;
#pragma unroll
        for (int i = 0; i < kHeads; ++i) {
          const float mn = fmaxf(fmaxf(mx[i], mr[i]), -1e30f);   // idle sub-groups stay finite
          const float p = valid ? expf(a[i] - mn) : 0.f;
#pragma unroll
          for (int m = 0; m < 6; ++m) v[i * 6 + m] = p * q[m];
          if (i == 0) scarg = mx[0] - mn;                     // -inf in the first round: exp -> 0
          mx[i] = mn;
        }
        float u[12], s6[6], w3[3];
#pragma unroll
        for (int t = 0; t < 12; ++t) u[t] = v[t] + __shfl_xor_sync(kFull, v[t + 12], 4);
#pragma unroll
        for (int t = 0; t < 6; ++t) s6[t] = u[t] + __shfl_xor_sync(kFull, u[t + 6], 2);
#pragma unroll
        for (int t = 0; t < 3; ++t) w3[t] = s6[t] + __shfl_xor_sync(kFull, s6[t + 3], 1);
        const float sc = expf(scarg);
#pragma unroll
        for (int t = 0; t < 3; ++t) acc3[t] = fmaf(acc3[t], sc, w3[t]);
      }
    }
    // even lane: sums x0..x2 of head sl>>1; odd lane: x3, x4 and the softmax denominator
    const float den_other = __shfl_xor_sync(kFull, acc3[2], 1);
    const float inv = 1.0f / ((odd ? acc3[2] : den_other) + 1e-16f);
    if constexpr (kHead) {
      // the row goes to the readout head of this CTA: slot (tile % 8) * 16 + graph of the group's buffer
      const int grp = k / kGroupTiles, buf = grp & 1, slot = (k % kGroupTiles) * kTG + gl;
      {
        ST_T1();
        st_wait(st_smem_u32(&sm.head.zfree[buf]), static_cast<unsigned>((grp >> 1) & 1) ^ 1u);   // group grp - 2 has been read
        ST_ACC1(4);
      }
      if (ok) {
        const int64_t l0 = st.ptrs[2][gl];
        float* zr = sm.head.zrow[buf] + slot * kZPitch + hx * kF + o0;
        zr[0] = acc3[0] * inv;
        zr[1] = acc3[1] * inv;
        if (!odd) zr[2] = acc3[2] * inv;
        if (sl == 0) {
          ti.d.lut_batch[l0] = ti.g0 + gl;
          ti.d.lut_node[l0] = static_cast<int32_t>(st.ptrs[0][gl]) + il;
          sm.head.optr[buf][slot] = ti.d.out + l0 * QOT_OUT;
        }
      } else if (sl == 0) {
        sm.head.optr[buf][slot] = nullptr;
      }
      __syncwarp();
      if (lane == 0) st_arrive(st_smem_u32(&sm.head.zfull[buf]));
    } else {
      if (ok) {
        const int64_t l0 = st.ptrs[2][gl];
        float* zr = ti.d.z + l0 * (kHeads * kF) + hx * kF + o0;
        zr[0] = acc3[0] * inv;
        zr[1] = acc3[1] * inv;
        if (!odd) zr[2] = acc3[2] * inv;
        if (sl == 0) {
          ti.d.lut_batch[l0] = ti.g0 + gl;
          ti.d.lut_node[l0] = static_cast<int32_t>(st.ptrs[0][gl]) + il;
        }
      }
    }
  }
  const bool generic = !ok && active && (!fits || (cnt == lrows && cnt > 0));
  const unsigned todo = __ballot_sync(kFull, generic && sl == 0);      // bit 8*s: graph s of this warp
  if (todo) {
    StGenericArgs& ga = gs.gargs;
    if (lane == 0) {
      ga.x = ti.d.x; ga.esrc = ti.d.edge_index; ga.edst = ti.d.edge_index + ti.d.E; ga.z = ti.d.z; ga.out = ti.d.out;
      ga.lut_batch = ti.d.lut_batch; ga.lut_node = ti.d.lut_node; ga.status = ti.d.status;
      ga.N = ti.d.N; ga.E = ti.d.E; ga.g0 = ti.g0 + gw * 4;
    }
    if (sl < 6) ga.p[sg][sl] = st.ptrs[sl >> 1][gl + (sl & 1)];
  }
  __syncwarp();
  if (lane == 0) st_arrive(ebar);                      // the x window is dead: the producer may refill the stage
  if (todo) {
    const unsigned t4 = (todo & 1u) | ((todo >> 7) & 2u) | ((todo >> 14) & 4u) | ((todo >> 21) & 8u);
    st_generic<kHead>(cw, t4, prep, lut_col, lane);
  }
}

// ------------------------------------------------------------------------------------------------
// in-kernel readout head (kHead): folded projection + BN + ReLU -> mlp.0 -> LeakyReLU -> mlp.3 for groups of 128 rows
//   epilogue warps 4..7: thread = row.  z (20 floats) from the staging buffer -> y = relu(z_h Wf_h + shift) on the FP32
//     pipe (640 FMA) -> split y = hi + lo (hi = the TF32 bits, lo = the exact remainder) -> tcgen05.st into TMEM as the
//     A operand of the next product: columns [0,128) hi, [128,256) lo.
//   MMA warp 1: one thread issues D[128x32] = A[128x128] * W1^T as 48 tcgen05.mma kind::tf32 (A from TMEM, B = the
//     swizzled mlp.0 weight in shared memory): hi*lo + lo*hi + hi*hi, fp32 accumulation in TMEM columns [256,288),
//     tcgen05.commit onto an mbarrier.
//   epilogue again: tcgen05.ld of the row's 32 hidden units, + b1, LeakyReLU, mlp.3 (96 FMA), 3 floats to out.
// The tensor pipe runs asynchronously beside the consumer warps: the head costs issue slots only for the epilogue.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long st_umma_desc_sw128(unsigned smem_addr) {
  // K-major, SWIZZLE_128B shared-memory matrix descriptor (as gemm_tc.cu): start address, LBO = 1, SBO = 1024 B,
  // version 1, layout type 2
  unsigned long long d = 0;
  d |= static_cast<unsigned long long>((smem_addr >> 4) & 0x3fffu);
  d |= static_cast<unsigned long long>(1u) << 16;
  d |= static_cast<unsigned long long>(1024u >> 4) << 32;
  d |= static_cast<unsigned long long>(1u) << 46;
  d |= static_cast<unsigned long long>(2u) << 61;
  return d;
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, N, M
constexpr unsigned st_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<unsigned>(N >> 3) << 17) | (static_cast<unsigned>(M >> 4) << 24);
}
__device__ __forceinline__ void st_umma_tf32_ts(unsigned tmem_d, unsigned tmem_a, unsigned long long bdesc, unsigned idesc,
                                                unsigned accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc),
      "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void st_tmem_st32(unsigned taddr, const unsigned (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void st_tmem_ld32(unsigned taddr, unsigned (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
constexpr unsigned kTmemCols = 512;        // columns [0,128) A hi, [128,256) A lo, [256,416) five accumulators
constexpr unsigned kTmemALo = 128, kTmemD = 256;

__device__ __noinline__ void st_head_mma(int ngroups, int lane) {
  StHeadSmem& hs = st_smem<true>().head;
  const unsigned tb = hs.tmem_base;
  constexpr unsigned idesc = st_idesc(128, 32);
  const unsigned b_hi = st_smem_u32(hs.b2[0]), b_lo = st_smem_u32(hs.b2[1]);
  for (int g = 0; g < ngroups; ++g) {
    if (!st_wait<200>(st_smem_u32(&hs.aready), static_cast<unsigned>(g & 1))) break;
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (lane == 0) {
      // five accumulators, summed in fp32 by the epilogue: the tensor core's add into a running accumulator truncates,
      // an error that grows linearly with the chain (csrc/gemm_tc.cu, profiles/r2_tc_chain_accuracy.md), so the large
      // hi*hi terms go to four short chains (4 steps = one 32-wide k-block each) and the two compensation products
      // (2^-11 of the magnitude, their truncation does not matter) to a fifth
#pragma unroll
      for (int p = 0; p < 3; ++p) {                   // hi*lo, lo*hi -> D4; hi*hi of k-block kb -> D[kb]
        const unsigned a_col = (p == 1) ? kTmemALo : 0u;
        const unsigned b_base = (p == 0) ? b_lo : b_hi;
#pragma unroll
        for (int kb = 0; kb < 4; ++kb)
#pragma unroll
          for (int s = 0; s < 4; ++s) {               // UMMA_K = 8 for tf32: 8 TMEM columns / 32 bytes of a swizzled row
            const unsigned d_col = p < 2 ? kTmemD + 128u : kTmemD + static_cast<unsigned>(kb * 32);
            const unsigned acc = p < 2 ? ((p | kb | s) != 0 ? 1u : 0u) : (s != 0 ? 1u : 0u);
            st_umma_tf32_ts(tb + d_col, tb + a_col + static_cast<unsigned>(kb * 32 + s * 8),
                            st_umma_desc_sw128(b_base + static_cast<unsigned>(kb * 4096 + s * 32)), idesc, acc);
          }
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                       st_smem_u32(&hs.dready))
                   : "memory");
    }
    __syncwarp();
  }
}

__device__ __noinline__ void st_head_epilogue(int my_tiles, int ngroups, int eq, int lane) {
  StHeadSmem& hs = st_smem<true>().head;
  const int row = eq * 32 + lane;
  const unsigned tb = hs.tmem_base + (static_cast<unsigned>(eq * 32) << 16);
  const float4* __restrict__ wf4 = reinterpret_cast<const float4*>(hs.wf);       // [h][f][32 channels]
  const float4* __restrict__ sh4 = reinterpret_cast<const float4*>(hs.shift);    // [128]
  ST_DECL();
  ST_T0();
  for (int g = 0; g < ngroups; ++g) {
    const int buf = g & 1;
    {
      ST_T1();
      if (!st_wait<200>(st_smem_u32(&hs.zfull[buf]), static_cast<unsigned>((g >> 1) & 1))) break;
      ST_ACC1(5);
    }
    float z[kHeads * kF];
    float* op = hs.optr[buf][row];
    if (g * kGroupTiles + (row >> 4) >= my_tiles) op = nullptr;      // slot of a tile past the CTA's last one
#pragma unroll
    for (int i = 0; i < kHeads * kF; ++i) z[i] = op ? hs.zrow[buf][row * kZPitch + i] : 0.f;
    __syncwarp();
    if (lane == 0) st_arrive(st_smem_u32(&hs.zfree[buf]));
#pragma unroll 1
    for (int h = 0; h < kHeads; ++h) {
      unsigned hi[32], lo[32];
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        float4 acc = sh4[h * 8 + c4];
#pragma unroll
        for (int f = 0; f < kF; ++f) {
          const float4 w = wf4[(h * kF + f) * 8 + c4];
          const float zf = z[h * kF + f];
          acc.x = fmaf(zf, w.x, acc.x); acc.y = fmaf(zf, w.y, acc.y);
          acc.z = fmaf(zf, w.z, acc.z); acc.w = fmaf(zf, w.w, acc.w);
        }
        const float y[4] = {fmaxf(acc.x, 0.f), fmaxf(acc.y, 0.f), fmaxf(acc.z, 0.f), fmaxf(acc.w, 0.f)};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // hi = the TF32 bits of y (truncation, exact: lo carries the rest); lo = the remainder + half a TF32 ulp,
          // so that the tensor core's own truncation of its low 13 bits rounds it to nearest instead of down
          const unsigned hb = __float_as_uint(y[j]) & 0xffffe000u;
          hi[c4 * 4 + j] = hb;
          lo[c4 * 4 + j] = __float_as_uint(y[j] - __uint_as_float(hb)) + 0x1000u;
        }
      }
      st_tmem_st32(tb + static_cast<unsigned>(h * 32), hi);
      st_tmem_st32(tb + kTmemALo + static_cast<unsigned>(h * 32), lo);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) st_arrive(st_smem_u32(&hs.aready));
    {
      ST_T1();
      if (!st_wait<100>(st_smem_u32(&hs.dready), static_cast<unsigned>(g & 1))) break;
      ST_ACC1(6);
    }
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    unsigned r[32];
    {
      unsigned r1[32], r2[32];
      st_tmem_ld32(tb + kTmemD, r);
      st_tmem_ld32(tb + kTmemD + 32u, r1);
      st_tmem_ld32(tb + kTmemD + 64u, r2);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        r[j] = __float_as_uint((__uint_as_float(r[j]) + __uint_as_float(r1[j])) + __uint_as_float(r2[j]));
      st_tmem_ld32(tb + kTmemD + 96u, r1);
      st_tmem_ld32(tb + kTmemD + 128u, r2);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        r[j] = __float_as_uint((__uint_as_float(r[j]) + __uint_as_float(r1[j])) + __uint_as_float(r2[j]));
    }
    float o3[QOT_OUT];
#pragma unroll
    for (int k = 0; k < QOT_OUT; ++k) o3[k] = hs.bo[k];
#pragma unroll
    for (int j4 = 0; j4 < 8; ++j4) {
      const float4 b1 = reinterpret_cast<const float4*>(hs.b1)[j4];
      float hv[4] = {__uint_as_float(r[4 * j4]) + b1.x, __uint_as_float(r[4 * j4 + 1]) + b1.y,
                     __uint_as_float(r[4 * j4 + 2]) + b1.z, __uint_as_float(r[4 * j4 + 3]) + b1.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) hv[j] = hv[j] > 0.f ? hv[j] : 0.01f * hv[j];
#pragma unroll
      for (int k = 0; k < QOT_OUT; ++k) {
        const float4 w2 = reinterpret_cast<const float4*>(hs.w2 + k * kHid)[j4];
        o3[k] = fmaf(hv[0], w2.x, o3[k]); o3[k] = fmaf(hv[1], w2.y, o3[k]);
        o3[k] = fmaf(hv[2], w2.z, o3[k]); o3[k] = fmaf(hv[3], w2.w, o3[k]);
      }
    }
    if (op) {
      op[0] = o3[0]; op[1] = o3[1]; op[2] = o3[2];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // this group's TMEM reads precede the next MMAs
  }
  ST_ACC(7);
  ST_FLUSH();
}

template <bool kHead, bool kSym>
__global__ void __launch_bounds__(StCfg<kHead>::kThreads, 1)
lp_stream_kernel(const qot_lp_batch_t* __restrict__ batches, int n_batches, int64_t tiles_per_batch,
                 int64_t total_tiles, const float* __restrict__ prep, int lut_col) {
  StSmemT<kHead>& sm = st_smem<kHead>();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int my_tiles = static_cast<int>((total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
  const int ngroups = (my_tiles + kGroupTiles - 1) / kGroupTiles;
  if (tid == 0) {
    for (int s = 0; s < StCfg<kHead>::kX; ++s) {
      st_mbar_init(&sm.full[s], 33);
      st_mbar_init(&sm.empty[s], kStGroupWarps);
    }
    for (int s = 0; s < StCfg<kHead>::kD; ++s) st_mbar_init(&sm.dempty[s], kStGroupWarps);
    if constexpr (kHead) {
      for (int i = 0; i < 2; ++i) {
        st_mbar_init(&sm.head.zfull[i], kGroupTiles * kStGroupWarps);
        st_mbar_init(&sm.head.zfree[i], 4);
      }
      st_mbar_init(&sm.head.aready, 4);
      st_mbar_init(&sm.head.dready, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    sm.next_unit = 0;
    sm.gen_lock = 0;
  }
  if (tid < 48) (&sm.asp[0][0])[tid] = __ldg(reinterpret_cast<const float4*>(prep + kOffAsP) + tid);
  if (tid >= 64 && tid < 64 + 4 * kF) (&sm.adp[0][0])[tid - 64] = __ldg(reinterpret_cast<const float4*>(prep + kOffAdP) + tid - 64);
  if constexpr (kHead) {
    float4* b2 = reinterpret_cast<float4*>(&sm.head.b2[0][0][0]);
    for (int i = tid; i < kB2swFloats / 4; i += StCfg<kHead>::kThreads)
      b2[i] = __ldg(reinterpret_cast<const float4*>(prep + kOffB2sw) + i);
    for (int i = tid; i < kHC * kF; i += StCfg<kHead>::kThreads) sm.head.wf[i] = __ldg(prep + kOffWf + i);
    if (tid < kHC) sm.head.shift[tid] = __ldg(prep + kOffShift + tid);
    if (tid < kHid) sm.head.b1[tid] = __ldg(prep + kOffB1 + tid);
    if (tid < QOT_OUT * kHid) sm.head.w2[tid] = __ldg(prep + kOffW2 + tid);
    if (tid < QOT_OUT) sm.head.bo[tid] = __ldg(prep + kOffB2 + tid);
    if (warp == 4) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(st_smem_u32(&sm.head.tmem_base)),
                   "r"(kTmemCols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the operand tile written above -> async proxy
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if constexpr (kHead) asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  if (warp == 0) {
    st_producer<kHead>(batches, n_batches, tiles_per_batch, batches[0].tile0, total_tiles, lane);
    return;
  }
  int cw = warp - 1;
  if constexpr (kHead) {
    if (warp == 1) {
      st_head_mma(ngroups, lane);
      return;
    }
    if (warp >= 4 && warp < 8) {
      st_head_epilogue(my_tiles, ngroups, warp - 4, lane);
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("bar.sync 1, 128;" ::: "memory");                  // the four epilogue warps: all TMEM reads done
      if (warp == 4)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(sm.head.tmem_base), "r"(kTmemCols) : "memory");
      return;
    }
    cw = warp < 4 ? warp - 2 : warp - 6;
  }
  // ---- consumers: every warp claims quarter-tiles (4 graphs) in order from one counter -- no static assignment,
  // so a slow quarter never idles another warp while stages hold data
  const int tiles_padded = kHead ? ngroups * kGroupTiles : my_tiles;
  ST_DECL();
  for (;;) {
    int u = 0;
    if (lane == 0) u = atomicAdd(&sm.next_unit, 1);
    u = __shfl_sync(kFull, u, 0);
    const int k = u >> 2, gw = u & 3;
    if (k >= tiles_padded) break;
    if constexpr (kHead) {
      if (k >= my_tiles) {
        // quarter of a tile past the last one: only the group protocol (its slots hold no rows)
        const int grp = k / kGroupTiles, buf = grp & 1;
        if (!st_wait(st_smem_u32(&sm.head.zfree[buf]), static_cast<unsigned>((grp >> 1) & 1) ^ 1u)) break;
        if (lane < 4) sm.head.optr[buf][(k % kGroupTiles) * kTG + gw * 4 + lane] = nullptr;
        __syncwarp();
        if (lane == 0) st_arrive(st_smem_u32(&sm.head.zfull[buf]));
        continue;
      }
    }
    const int s = k % StCfg<kHead>::kX;
    const unsigned ph = static_cast<unsigned>((k / StCfg<kHead>::kX) & 1);
    {
      ST_T0();
      if (!st_wait(st_smem_u32(&sm.full[s]), ph)) {
        if (lane == 0) atomicOr(batches[0].status, 4);
        break;
      }
      ST_ACC(2);
    }
    ST_T0();
    st_consume_tile<kHead, kSym>(k, cw, prep, lut_col, gw, lane ST_ARG);
    ST_ACC(3);
  }
  ST_FLUSH();
}

// ------------------------------------------------------------------------------------------------
// readout head over the z rows of every batch of the launch (grid.y = batch): folded projection + BN + ReLU
// -> mlp.0 -> LeakyReLU -> mlp.3 on the tensor cores (mma.sync TF32 x3), 64 rows per block
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
lp_stream_head_kernel(const qot_lp_batch_t* __restrict__ batches, const float* __restrict__ prep) {
  __shared__ float4 frag[kStHeadFrag4];
  const qot_lp_batch_t& d = batches[blockIdx.y];
  const float* __restrict__ zbuf = d.z;
  float* __restrict__ out = d.out;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g8 = lane >> 2, t4 = lane & 3;
  const int64_t L = d.lut_ptr[d.B];
  if (static_cast<int64_t>(blockIdx.x) * 64 >= L) return;
  for (int i = tid; i < kStHeadFrag4; i += 128) frag[i] = __ldg(reinterpret_cast<const float4*>(prep + kOffB1f) + i);
  __syncthreads();
  const float4* __restrict__ f1 = frag;
  const float4* __restrict__ f2 = frag + 16 * 32;
  for (int64_t tile = static_cast<int64_t>(blockIdx.x) * 4 + warp; tile * 16 < L;
       tile += static_cast<int64_t>(gridDim.x) * 4) {
    const int64_t ra = tile * 16 + g8, rb = ra + 8;
    const bool va = ra < L, vb = rb < L;
    float oa, ob;
    head_rows16_tf32x3(f1, f2, zbuf + ra * (kHeads * kF), zbuf + rb * (kHeads * kF), va, vb, prep, lane, oa, ob);
    if (t4 < QOT_OUT) {
      if (va) out[ra * QOT_OUT + t4] = oa;
      if (vb) out[rb * QOT_OUT + t4] = ob;
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Compact wire format of a verified-layout batch (what travels over PCIe; qot_lightpath_infer_wire_host):
//   int32 ptr[B+1] | int32 edge_ptr[B+1] | int32 lut_ptr[B+1] | pad16 | float x4[N,4] | pad16 | uint8 lut_local[L] | pad16
//   | uint8 dst[E]
// x4 = the four node features other than the LUT flag (the flag column holds exactly 0.0 / 1.0 -- checked when the
// batch is packed -- so it travels as lut_local: the graph-local node index of every readout row, in row order);
// dst = the destination of every edge as a GRAPH-LOCAL id (graphs of <= 255 nodes); no source row: under the
// verified from_networkx layout (QOT_LP_SYMMETRIC_BY_SOURCE) the out-run of node u is edges
// [#{dst < u}, #{dst <= u}) of its graph, so the sources are the run index.  649 B/graph at n = 32, E_g = 124
// against 1 754 B/graph for the int64 destination row + offsets + x.
// lp_wire_unpack_kernel rebuilds the reference layout ON THE DEVICE (x [N,5], int64 edge_index [2,E] with batch-global
// ids, int64 ptr / edge_ptr / lut_ptr) and fills the sizes of the slot's batch descriptor; the
// batch then goes through the same lp_stream_kernel as a resident batch (bit-identical rows).  One warp per graph.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
lp_wire_unpack_kernel(const int32_t* __restrict__ wptr, const int32_t* __restrict__ weptr, const int32_t* __restrict__ wlptr,
                      const uint8_t* __restrict__ wdst, const float* __restrict__ x4, const uint8_t* __restrict__ wlut,
                      int lut_col, int64_t N, int64_t E, int64_t B, int64_t L, int64_t* __restrict__ ptrs,
                      int64_t* __restrict__ edge_index, qot_lp_batch_t* __restrict__ desc, float* __restrict__ x,
                      char* __restrict__ result) {
  __shared__ int hist[8][257];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t gtid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  for (int64_t i = gtid; i < 3 * (B + 1); i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t which = i / (B + 1), j = i % (B + 1);
    ptrs[i] = (which == 0 ? wptr : which == 1 ? weptr : wlptr)[j];
  }
  if (gtid == 0) {
    desc->x = x;
    desc->edge_index = edge_index;
    desc->ptr = ptrs; desc->edge_ptr = ptrs + (B + 1); desc->lut_ptr = ptrs + 2 * (B + 1);
    desc->N = N; desc->E = E; desc->B = B;
    desc->tile0 = 0;
    // result arena of the slot: [status, 16 bytes | out [L,3] | pad to 16 | lut_batch [L]] -- ONE device->host copy
    desc->status = reinterpret_cast<int32_t*>(result);
    desc->out = reinterpret_cast<float*>(result + 16);
    desc->lut_batch = reinterpret_cast<int64_t*>(result + 16 + ((12 * L + 15) & ~15ll));
  }
  int* h = hist[w];
  for (int64_t g = blockIdx.x * 8ll + w; g < B; g += static_cast<int64_t>(gridDim.x) * 8) {
    const int n0 = wptr[g], n = wptr[g + 1] - n0, e0 = weptr[g], ne = weptr[g + 1] - e0;
    if (n < 0 || n > 255 || ne < 0 || e0 < 0 || static_cast<int64_t>(e0) + ne > E) {
      if (lane == 0) atomicOr(reinterpret_cast<int32_t*>(result), 1);   // malformed offsets: nothing is written for the graph
      continue;
    }
    // node features: the four shipped columns around a LUT flag column of zeros, then 1.0 at the readout rows
    for (int i = lane; i < n * kF; i += 32) {
      const int node = i / kF, c = i % kF;
      x[static_cast<int64_t>(n0) * kF + i] = c == lut_col ? 0.f : x4[(static_cast<int64_t>(n0) + node) * 4 + (c - (c > lut_col))];
    }
    __syncwarp();
    for (int r = wlptr[g] + lane; r < wlptr[g + 1]; r += 32) {
      const int li = wlut[r];
      if (li < n) x[(static_cast<int64_t>(n0) + li) * kF + lut_col] = 1.0f; else atomicOr(reinterpret_cast<int32_t*>(result), 1);
    }
    for (int i = lane; i <= n; i += 32) h[i] = 0;
    __syncwarp();
    for (int i = lane; i < ne; i += 32) {
      const int d = wdst[e0 + i];
      edge_index[E + e0 + i] = n0 + d;                               // destination row
      if (d < n) atomicAdd(&h[d + 1], 1); else atomicOr(reinterpret_cast<int32_t*>(result), 1);
    }
    __syncwarp();
    // exclusive prefix of the in-degree (= out-degree) histogram: h[u] = first edge of node u's run
    int carry = 0;
    for (int b0 = 0; b0 <= n; b0 += 32) {
      const int i = b0 + lane;
      int v = i <= n ? h[i] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(kFull, v, o);
        if (lane >= o) v += up;
      }
      if (i <= n) h[i] = v + carry;
      carry += __shfl_sync(kFull, v, 31);
    }
    __syncwarp();
    for (int u = lane; u < n; u += 32)
      for (int e = h[u]; e < h[u + 1] && e < ne; ++e) edge_index[e0 + e] = n0 + u;   // source row
    __syncwarp();
  }
}

}  // namespace qot

using namespace qot;

#ifdef QOT_ST_TRACE
extern "C" int qot_debug_set_st_trace(unsigned long long* buf) {
  return cudaMemcpyToSymbol(g_st_trace, &buf, sizeof(buf)) == cudaSuccess ? 0 : -3;
}
#endif

extern "C" int64_t qot_lightpath_stream_tiles(int64_t B) { return B > 0 ? cdiv(B, kTG) : 0; }

// `batches`: DEVICE array of n_batches descriptors with tile0 filled (tile0[b+1] = tile0[b] +
// qot_lightpath_stream_tiles(B_b); tile0[0] is arbitrary, so a sub-range of a longer array can be launched);
// total_tiles = the tiles of these batches; uniform_tiles = tiles per batch when every batch but the last has
// the same count (0: the kernel searches tile0).  max_rows = the largest lut_ptr[B] over
// the batches (an upper bound such as max N is fine): sizes the head grid.  The status words of the batches
// must be zero on entry (one cudaMemsetAsync over a pooled array does it).
extern "C" int qot_lightpath_infer_stream(const qot_lp_batch_t* batches, int32_t n_batches, int64_t total_tiles,
                                          int64_t uniform_tiles, int64_t max_rows, const float* prepared,
                                          int32_t is_lut_index, int32_t flags, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  QOT_REQUIRE(batches && n_batches > 0 && total_tiles >= 0 && uniform_tiles >= 0 && max_rows >= 0,
              "qot_lightpath_infer_stream: bad argument");
  QOT_REQUIRE(prepared && (reinterpret_cast<uintptr_t>(prepared) & 15) == 0,
              "qot_lightpath_infer_stream: prepared must be 16-byte aligned");
  QOT_REQUIRE(is_lut_index >= 0 && is_lut_index < kF, "qot_lightpath_infer_stream: is_lut_index out of range");
  if (total_tiles == 0) return QOT_OK;
  QOT_REQUIRE((flags & ~(QOT_LP_SYMMETRIC_BY_SOURCE | QOT_LP_SPLIT_HEAD)) == 0, "qot_lightpath_infer_stream: unknown flag");
  const bool sym = (flags & QOT_LP_SYMMETRIC_BY_SOURCE) != 0, split = (flags & QOT_LP_SPLIT_HEAD) != 0;
  static std::atomic<unsigned long long> done{0};
  constexpr int smem_split = static_cast<int>(sizeof(StSmemT<false>) + 1024), smem_head = static_cast<int>(sizeof(StSmemT<true>) + 1024);
  if (int rc = once_per_device(done, [] {
        QOT_CUDA(cudaFuncSetAttribute(lp_stream_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_split));
        QOT_CUDA(cudaFuncSetAttribute(lp_stream_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_split));
        QOT_CUDA(cudaFuncSetAttribute(lp_stream_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_head));
        QOT_CUDA(cudaFuncSetAttribute(lp_stream_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_head));
        return static_cast<int>(QOT_OK);
      }))
    return rc;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(kNumSMs, total_tiles));
  if (!split) {
    if (sym)
      lp_stream_kernel<true, true><<<grid, StCfg<true>::kThreads, smem_head, stream>>>(batches, n_batches, uniform_tiles,
                                                                                   total_tiles, prepared, is_lut_index);
    else
      lp_stream_kernel<true, false><<<grid, StCfg<true>::kThreads, smem_head, stream>>>(batches, n_batches, uniform_tiles,
                                                                                    total_tiles, prepared, is_lut_index);
    QOT_LAUNCH_CHECK();
    return QOT_OK;
  }
  if (sym)
    lp_stream_kernel<false, true><<<grid, StCfg<false>::kThreads, smem_split, stream>>>(batches, n_batches, uniform_tiles,
                                                                                     total_tiles, prepared, is_lut_index);
  else
    lp_stream_kernel<false, false><<<grid, StCfg<false>::kThreads, smem_split, stream>>>(batches, n_batches, uniform_tiles,
                                                                                      total_tiles, prepared, is_lut_index);
  QOT_LAUNCH_CHECK();
  const int64_t hb = std::max<int64_t>(1, std::min<int64_t>(cdiv(max_rows, 64), 4 * kNumSMs));
  lp_stream_head_kernel<<<dim3(static_cast<unsigned>(hb), static_cast<unsigned>(n_batches)), 128, 0, stream>>>(batches, prepared);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}

static inline size_t wire_align16(size_t v) { return (v + 15) & ~size_t(15); }
extern "C" size_t qot_lightpath_wire_bytes(int64_t N, int64_t E, int64_t B, int64_t L) {
  if (N < 0 || E < 0 || B < 0 || L < 0) return 0;
  return wire_align16(12 * static_cast<size_t>(B + 1)) + wire_align16(16 * static_cast<size_t>(N)) + wire_align16(static_cast<size_t>(L)) +
         wire_align16(static_cast<size_t>(E));
}

extern "C" size_t qot_lightpath_wire_result_bytes(int64_t L) {
  return L < 0 ? 0 : 16 + wire_align16(12 * static_cast<size_t>(L)) + 8 * static_cast<size_t>(L);
}

// One batch from PINNED HOST memory in the compact wire format, end to end on `stream`: ONE host->device copy of the
// arena, lp_wire_unpack_kernel, lp_stream_kernel over the slot's descriptor, ONE device->host copy of the result arena
// [status | out rows | lut_batch rows] (L = the batch's readout rows, known on the host: lut_ptr[B]).  Nothing
// synchronises; the caller waits on its own event.  The slot is caller-owned device memory (see qot_lp_wire_slot_t).
extern "C" int qot_lightpath_infer_wire_host(const void* arena_host, int64_t N, int64_t E, int64_t B, int64_t L,
                                             const float* prepared, int32_t is_lut_index, const qot_lp_wire_slot_t* slot,
                                             void* result_host, int64_t* h2d_bytes, int64_t* d2h_bytes, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  QOT_REQUIRE(arena_host && slot && prepared && result_host, "qot_lightpath_infer_wire_host: null argument");
  QOT_REQUIRE(N > 0 && B > 0 && E >= 0 && L >= 0 && L <= N, "qot_lightpath_infer_wire_host: bad size");
  QOT_REQUIRE(slot->arena && slot->x && slot->edge_index && slot->ptrs && slot->desc && slot->result && slot->lut_node &&
                  slot->n_lut, "qot_lightpath_infer_wire_host: incomplete staging slot");
  QOT_REQUIRE(is_lut_index >= 0 && is_lut_index < kF, "qot_lightpath_infer_wire_host: is_lut_index out of range");
  QOT_REQUIRE(N <= slot->cap_nodes && E <= slot->cap_edges && B <= slot->cap_graphs,
              "qot_lightpath_infer_wire_host: batch (N=%lld, E=%lld, B=%lld) exceeds the slot capacity", (long long)N,
              (long long)E, (long long)B);
  QOT_REQUIRE((reinterpret_cast<uintptr_t>(slot->arena) & 15) == 0 && (reinterpret_cast<uintptr_t>(slot->desc) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(slot->result) & 15) == 0,
              "qot_lightpath_infer_wire_host: slot arena / descriptor / result must be 16-byte aligned");
  const size_t nbytes = qot_lightpath_wire_bytes(N, E, B, L), rbytes = qot_lightpath_wire_result_bytes(L);
  QOT_CUDA(cudaMemcpyAsync(slot->arena, arena_host, nbytes, cudaMemcpyHostToDevice, stream));
  const char* a = static_cast<const char*>(slot->arena);
  const int32_t* wptr = reinterpret_cast<const int32_t*>(a);
  const size_t o_x = wire_align16(12 * static_cast<size_t>(B + 1)), o_l = o_x + wire_align16(16 * static_cast<size_t>(N)),
               o_d = o_l + wire_align16(static_cast<size_t>(L));
  const float* x4 = reinterpret_cast<const float*>(a + o_x);
  const uint8_t* wlut = reinterpret_cast<const uint8_t*>(a + o_l);
  const uint8_t* wdst = reinterpret_cast<const uint8_t*>(a + o_d);
  QOT_CUDA(cudaMemsetAsync(slot->result, 0, 16, stream));           // the status word
  const unsigned ub = static_cast<unsigned>(std::min<int64_t>(cdiv(B, 8), 4 * kNumSMs));
  lp_wire_unpack_kernel<<<ub, 256, 0, stream>>>(wptr, wptr + (B + 1), wptr + 2 * (B + 1), wdst, x4, wlut, is_lut_index, N, E, B, L,
                                               slot->ptrs, slot->edge_index, slot->desc, slot->x,
                                               static_cast<char*>(slot->result));
  QOT_LAUNCH_CHECK();
  const int64_t tiles = qot_lightpath_stream_tiles(B);
  int rc = qot_lightpath_infer_stream(slot->desc, 1, tiles, tiles, L, prepared, is_lut_index, QOT_LP_SYMMETRIC_BY_SOURCE, stream_);
  if (rc) return rc;
  QOT_CUDA(cudaMemcpyAsync(result_host, slot->result, rbytes, cudaMemcpyDeviceToHost, stream));
  if (h2d_bytes) *h2d_bytes = static_cast<int64_t>(nbytes);
  if (d2h_bytes) *d2h_bytes = static_cast<int64_t>(rbytes);
  return QOT_OK;
}
