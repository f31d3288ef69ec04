// Device helpers shared by the LightpathGNN eval sources (lightpath_infer.cu: parameter folding and lut_ptr;
// lightpath_stream.cu: the persistent kernel; lightpath_every_node.cu: every node as the LUT):
// layout of the prepared parameter block, TF32 split helpers, the warp-per-row attention used by
// the generic path, the FP32 readout head of one row, the mma.sync readout head of 16 rows.
#pragma once
#include "common.cuh"

namespace qot {


// prepared-parameter layout (floats)
constexpr int kF = QOT_GAT_IN;       // 5
constexpr int kHeads = QOT_GAT_HEADS;  // 4
constexpr int kC = QOT_GAT_C;        // 32
constexpr int kHC = QOT_GAT_HC;      // 128
constexpr int kHid = 32;             // mlp hidden
constexpr int kOffAsrc = 0;                       // [f][h] 20
constexpr int kOffAdst = kOffAsrc + kF * kHeads;  // [f][h] 20
constexpr int kOffWf = kOffAdst + kF * kHeads;    // [h][f][c%32] 640, BN scale folded in
constexpr int kOffShift = kOffWf + kHC * kF;      // [c] 128 (conv bias + BN folded)
constexpr int kOffW1t = kOffShift + kHC;          // [c][o] 4096
constexpr int kOffB1 = kOffW1t + kHC * kHid;      // [o] 32
constexpr int kOffW2 = kOffB1 + kHid;             // [k][o] 96
constexpr int kOffB2 = kOffW2 + QOT_OUT * kHid;   // [k] 3
constexpr int kPreparedBase = ((kOffB2 + QOT_OUT + 3) / 4) * 4;
// tensor-core operand fragments of the readout head (lp_infer_bulk_kernel): every entry is a float4
// {b0_hi, b1_hi, b0_lo, b1_lo} of one lane of an m16n8k8 TF32 B fragment, hi = round-to-TF32, lo = TF32
// of the residual (error-compensated 3-product scheme, as in gemm_tc.cu)
constexpr int kOffB1f = kPreparedBase;                  // [ntile 16][lane 32][4]: folded GAT projection + shift row
constexpr int kOffB2f = kOffB1f + 16 * 32 * 4;          // [ktile 16][ntile 4][lane 32][4]: mlp.0 weight
// attention vectors in the per-lane slot order of lp_attn_kernel (see there)
constexpr int kOffAsP = kOffB2f + 16 * 4 * 32 * 4;      // [sl 8][slot 6][head slot 4]
constexpr int kOffAdP = kOffAsP + 8 * 6 * 4;            // [sl>>1 4][f 5][head slot 4]
// mlp.0 weight as the B operand of tcgen05.mma kind::tf32 (lp_stream_kernel's readout head): [hi | lo][k-block 4]
// [row n 32][32 floats], K-major with the 128-byte swizzle the UMMA shared-memory descriptor names (16-byte chunk c of
// row n stored at chunk c ^ (n & 7)); hi = round-to-TF32, lo = TF32 of the residual.  4096-byte aligned in `prepared`.
constexpr int kOffB2sw = ((kOffAdP + 4 * kF * 4 + 1023) / 1024) * 1024;
constexpr int kB2swFloats = 2 * 4 * 32 * 32;
constexpr int kPreparedFloats = kOffB2sw + kB2swFloats;

__device__ __forceinline__ unsigned tf32_rna(float v) {
  unsigned r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return r;
}
// the same rounding for finite inputs (cvt.rna.tf32 is add-half-ulp + mask plus an Inf/NaN guard on sm_100)
__device__ __forceinline__ unsigned tf32_rna_finite(float v) { return (__float_as_uint(v) + 0x1000u) & 0xffffe000u; }
__device__ __forceinline__ float4 tf32_split2(float b0, float b1) {
  const float h0 = __uint_as_float(tf32_rna(b0)), h1 = __uint_as_float(tf32_rna(b1));
  return make_float4(h0, h1, __uint_as_float(tf32_rna(b0 - h0)), __uint_as_float(tf32_rna(b1 - h1)));
}

constexpr int kMaxN = 64;                 // fast path: nodes of a graph staged in shared memory
constexpr int kMsgCap = 64;               // message list per warp (sources of one row + its self loop)

__device__ __forceinline__ float pick5(const float (&v)[kF], int f) {
  return (f == 0) ? v[0] : (f == 1) ? v[1] : (f == 2) ? v[2] : (f == 3) ? v[3] : v[4];
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Attention over a list of message sources, 8 messages per round: lane = (slot m = lane>>2,
// head h = lane&3).  Online softmax across rounds; within a round the 8 slots are combined by
// a fixed xor-shuffle tree, so the result depends only on the (edge-ordered) list.
struct AttnState {
  float m = -INFINITY, ssum = 0.f, acc[kF] = {0.f, 0.f, 0.f, 0.f, 0.f};
};
template <typename XF>
__device__ __forceinline__ void attn_consume(AttnState& st, const int* msg, int M, XF xf,
                                             const float (&As)[kF], float d_i, int lane) {
  const int slot = lane >> 2;
  for (int r0 = 0; r0 < M; r0 += 8) {
    const bool valid = r0 + slot < M;
    const int j = msg[valid ? r0 + slot : r0];
    float xj[kF];
#pragma unroll
    for (int k = 0; k < kF; ++k) xj[k] = xf(j, k);
    float a = d_i;
#pragma unroll
    for (int k = 0; k < kF; ++k) a = fmaf(xj[k], As[k], a);
    a = a > 0.f ? a : 0.2f * a;                     // leaky_relu(., 0.2)
    if (!valid) a = -INFINITY;
    float mr = a;
#pragma unroll
    for (int o = 4; o <= 16; o <<= 1) mr = fmaxf(mr, __shfl_xor_sync(kFull, mr, o));
    const float mn = fmaxf(st.m, mr);               // finite: slot 0 of every round is valid
    const float sc = expf(st.m - mn);               // exp(-inf) = 0 in the first round
    const float p = valid ? expf(a - mn) : 0.f;
    float v[kF + 1];
    v[kF] = p;
#pragma unroll
    for (int k = 0; k < kF; ++k) v[k] = p * xj[k];
#pragma unroll
    for (int o = 4; o <= 16; o <<= 1) {
#pragma unroll
      for (int k = 0; k <= kF; ++k) v[k] += __shfl_xor_sync(kFull, v[k], o);
    }
    st.ssum = fmaf(st.ssum, sc, v[kF]);
#pragma unroll
    for (int k = 0; k < kF; ++k) st.acc[k] = fmaf(st.acc[k], sc, v[k]);
    st.m = mn;
  }
}
// z[h][f] = acc / (sum + 1e-16) into slot h*kPitch+f of s_z (lane (m,h) stores feature m)
template <int kPitch = 8>
__device__ __forceinline__ void attn_finish(const AttnState& st, float* s_z, int lane) {
  const int slot = lane >> 2, h = lane & 3;
  const float den = st.ssum + 1e-16f;
  if (slot < kF) s_z[h * kPitch + slot] = pick5(st.acc, slot) / den;
}

// z (slot h*8+f of s_z) -> folded projection + BatchNorm + ReLU -> MLP head; lanes 0..2 return out[k].
// `w` = the prepared block from kOffWf on (shared memory in the kernel).
__device__ __forceinline__ float lut_row_head(const float* __restrict__ w, const float* s_z, float* s_y,
                                              int lane) {
  constexpr int oShift = kOffShift - kOffWf, oW1 = kOffW1t - kOffWf, oB1 = kOffB1 - kOffWf,
                oW2 = kOffW2 - kOffWf, oB2 = kOffB2 - kOffWf;
  // y[c], c = h2*32 + lane
#pragma unroll
  for (int h2 = 0; h2 < kHeads; ++h2) {
    float v = w[oShift + h2 * kC + lane];
#pragma unroll
    for (int k = 0; k < kF; ++k) v = fmaf(w[(h2 * kF + k) * kC + lane], s_z[h2 * 8 + k], v);
    s_y[h2 * kC + lane] = fmaxf(v, 0.f);
  }
  __syncwarp();
  // hidden layer: lane = (cg, og) owns outputs 4og..4og+3 over channels [32cg, 32cg+32)
  const int cg = lane >> 3, og = lane & 7;
  const float4* __restrict__ w1 = reinterpret_cast<const float4*>(w + oW1) + cg * 32 * (kHid / 4) + og;
  const float4* __restrict__ yq = reinterpret_cast<const float4*>(s_y + cg * 32);
  float4 h4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) {
    const float4 yv = yq[c4];
    const float4 wa = w1[(4 * c4 + 0) * (kHid / 4)];
    const float4 wb = w1[(4 * c4 + 1) * (kHid / 4)];
    const float4 wc = w1[(4 * c4 + 2) * (kHid / 4)];
    const float4 wd = w1[(4 * c4 + 3) * (kHid / 4)];
    h4.x = fmaf(wa.x, yv.x, h4.x); h4.y = fmaf(wa.y, yv.x, h4.y); h4.z = fmaf(wa.z, yv.x, h4.z); h4.w = fmaf(wa.w, yv.x, h4.w);
    h4.x = fmaf(wb.x, yv.y, h4.x); h4.y = fmaf(wb.y, yv.y, h4.y); h4.z = fmaf(wb.z, yv.y, h4.z); h4.w = fmaf(wb.w, yv.y, h4.w);
    h4.x = fmaf(wc.x, yv.z, h4.x); h4.y = fmaf(wc.y, yv.z, h4.y); h4.z = fmaf(wc.z, yv.z, h4.z); h4.w = fmaf(wc.w, yv.z, h4.w);
    h4.x = fmaf(wd.x, yv.w, h4.x); h4.y = fmaf(wd.y, yv.w, h4.y); h4.z = fmaf(wd.z, yv.w, h4.z); h4.w = fmaf(wd.w, yv.w, h4.w);
  }
#pragma unroll
  for (int o = 8; o <= 16; o <<= 1) {
    h4.x += __shfl_xor_sync(kFull, h4.x, o);
    h4.y += __shfl_xor_sync(kFull, h4.y, o);
    h4.z += __shfl_xor_sync(kFull, h4.z, o);
    h4.w += __shfl_xor_sync(kFull, h4.w, o);
  }
  const float4 b1 = reinterpret_cast<const float4*>(w + oB1)[og];
  float4 act = make_float4(h4.x + b1.x, h4.y + b1.y, h4.z + b1.z, h4.w + b1.w);
  act.x = act.x > 0.f ? act.x : 0.01f * act.x;
  act.y = act.y > 0.f ? act.y : 0.01f * act.y;
  act.z = act.z > 0.f ? act.z : 0.01f * act.z;
  act.w = act.w > 0.f ? act.w : 0.01f * act.w;
  float o3[QOT_OUT];
#pragma unroll
  for (int k = 0; k < QOT_OUT; ++k) {
    const float4 wk = reinterpret_cast<const float4*>(w + oW2 + k * kHid)[og];
    o3[k] = wk.x * act.x + wk.y * act.y + wk.z * act.z + wk.w * act.w;
  }
#pragma unroll
  for (int o = 1; o <= 4; o <<= 1) {
#pragma unroll
    for (int k = 0; k < QOT_OUT; ++k) o3[k] += __shfl_xor_sync(kFull, o3[k], o);
  }
  const float b2 = lane < QOT_OUT ? w[oB2 + lane] : 0.f;
  return (lane == 0 ? o3[0] : lane == 1 ? o3[1] : o3[2]) + b2;
}

// x accessors of the generic row: XRaw reads x as stored; XAsLut reads it with the LUT flag column overridden --
// 1.0 for node `lut` and 0.0 for every other node (every-node mode: row `lut` evaluated as the LUT)
struct XRaw {
  const float* __restrict__ x;
  __device__ __forceinline__ float operator()(int64_t j, int k) const { return x[j * kF + k]; }
};
struct XAsLut {
  const float* __restrict__ x;
  int64_t lut;
  int col;
  __device__ __forceinline__ float operator()(int64_t j, int k) const {
    return k == col ? (j == lut ? 1.0f : 0.0f) : x[j * kF + k];
  }
};

// Generic row evaluation straight from global memory: graphs beyond the fast-path caps, further
// LUT rows of a graph, rows with more than kMsgCap-1 in-edges or a source outside their slab.
// kHead = false: z only, into slot h*8+f of s_z.
template <bool kHead = true, typename XF = XRaw>
__device__ __noinline__ float lut_row_global(XF xg, const int64_t* __restrict__ esrc,
                                             const int64_t* __restrict__ edst, int64_t e0, int64_t e1,
                                             int64_t N, int64_t i, const float* __restrict__ prep,
                                             const float* __restrict__ w, int* s_msg, float* s_z,
                                             float* s_y, int lane) {
  const int h = lane & 3;
  float As[kF], d_i = 0.f;
#pragma unroll
  for (int k = 0; k < kF; ++k) {
    As[k] = __ldg(prep + kOffAsrc + k * kHeads + h);
    d_i = fmaf(xg(i, k), __ldg(prep + kOffAdst + k * kHeads + h), d_i);
  }
  auto xf = [&](int j, int k) { return xg(static_cast<int64_t>(j), k); };
  AttnState st;
  int cnt = 0;
  for (int64_t eb = e0; eb < e1; eb += 32) {
    const int64_t e = eb + lane;
    const int64_t dd = (e < e1) ? edst[e] : -1;
    int64_t sj = i;
    if (dd == i) sj = esrc[e];
    const bool hit = (dd == i) && (sj != i) && (static_cast<uint64_t>(sj) < static_cast<uint64_t>(N));
    const unsigned hm = __ballot_sync(kFull, hit);
    if (hit) s_msg[cnt + __popc(hm & ((1u << lane) - 1u))] = static_cast<int>(sj);
    cnt += __popc(hm);
    if (cnt >= kMsgCap - 32) {                                   // warp-uniform: keep room for 32 more
      __syncwarp();
      attn_consume(st, s_msg, cnt, xf, As, d_i, lane);
      __syncwarp();
      cnt = 0;
    }
  }
  if (lane == 0) s_msg[cnt] = static_cast<int>(i);               // the appended self loop comes last
  ++cnt;
  __syncwarp();
  attn_consume(st, s_msg, cnt, xf, As, d_i, lane);
  attn_finish(st, s_z, lane);
  __syncwarp();
  if (!kHead) return 0.f;                                        // z only (lp_attn_kernel)
  const float ov = lut_row_head(w, s_z, s_y, lane);
  __syncwarp();
  return ov;
}

// ------------------------------------------------------------------------------------------------
// readout head of 16 z rows on the tensor cores (mma.sync m16n8k8 TF32, split-fp32 operands: hi*lo + lo*hi
// + hi*hi), one warp: folded projection + BN + ReLU -> mlp.0 -> LeakyReLU -> mlp.3.  Row g8 = lane >> 2 of the
// tile is `za` (20 floats, [h][f]), row g8 + 8 is `zb`; `va` / `vb`: the row exists (else zeros go in).  `f1` /
// `f2`: the B1f / B2f fragment tables of `prepared` (kStHeadFrag4 float4, shared memory in the kernels).
// Lanes t4 = lane & 3 < 3 return output t4 of both rows in oa / ob.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_mma_tf32(float (&c)[4], const unsigned (&a)[4], float b0, float b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}
constexpr int kStHeadFrag4 = (kOffAsP - kOffB1f) / 4;   // float4 entries of B1f | B2f (contiguous in `prepared`)

__device__ __forceinline__ void head_rows16_tf32x3(const float4* __restrict__ f1, const float4* __restrict__ f2,
                                                   const float* za, const float* zb, bool va, bool vb,
                                                   const float* __restrict__ prep, int lane, float& oa_out,
                                                   float& ob_out) {
  const int t4 = lane & 3;
  float H[4][4], Hc[4][4];                             // fp32 sums of the hi x hi tiles; compensation chains
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int i = 0; i < 4; ++i) H[q][i] = Hc[q][i] = 0.f;
#pragma unroll 1
  for (int h = 0; h < kHeads; ++h) {
    unsigned ahi[4], alo[4];
    {
      float a[4];
      a[0] = va ? za[h * kF + t4] : 0.f;
      a[1] = vb ? zb[h * kF + t4] : 0.f;
      a[2] = t4 == 0 ? (va ? za[h * kF + 4] : 0.f) : (t4 == 1 ? 1.0f : 0.f);
      a[3] = t4 == 0 ? (vb ? zb[h * kF + 4] : 0.f) : (t4 == 1 ? 1.0f : 0.f);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        ahi[i] = tf32_rna(a[i]);
        alo[i] = tf32_rna(a[i] - __uint_as_float(ahi[i]));
      }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int j = 4 * h + jj;
      const float4 b = f1[j * 32 + lane];
      float c[4] = {0.f, 0.f, 0.f, 0.f};
      st_mma_tf32(c, alo, b.x, b.y);
      st_mma_tf32(c, ahi, b.z, b.w);
      st_mma_tf32(c, ahi, b.x, b.y);
      const float y[4] = {fmaxf(c[0], 0.f), fmaxf(c[2], 0.f), fmaxf(c[1], 0.f), fmaxf(c[3], 0.f)};
      unsigned yhi[4], ylo[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        yhi[i] = tf32_rna_finite(y[i]);
        ylo[i] = tf32_rna_finite(y[i] - __uint_as_float(yhi[i]));
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b2 = f2[(j * 4 + q) * 32 + lane];
        st_mma_tf32(Hc[q], ylo, b2.x, b2.y);
        st_mma_tf32(Hc[q], yhi, b2.z, b2.w);
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        st_mma_tf32(t, yhi, b2.x, b2.y);
#pragma unroll
        for (int i = 0; i < 4; ++i) H[q][i] += t[i];
      }
    }
  }
  float oa[QOT_OUT] = {0.f, 0.f, 0.f}, ob[QOT_OUT] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int o = 8 * q + 2 * t4;
    const float2 b1 = __ldg(reinterpret_cast<const float2*>(prep + kOffB1 + o));
    float hv[4] = {H[q][0] + Hc[q][0] + b1.x, H[q][1] + Hc[q][1] + b1.y, H[q][2] + Hc[q][2] + b1.x,
                   H[q][3] + Hc[q][3] + b1.y};
#pragma unroll
    for (int i = 0; i < 4; ++i) hv[i] = hv[i] > 0.f ? hv[i] : 0.01f * hv[i];
#pragma unroll
    for (int k = 0; k < QOT_OUT; ++k) {
      const float2 w2 = __ldg(reinterpret_cast<const float2*>(prep + kOffW2 + k * kHid + o));
      oa[k] = fmaf(hv[0], w2.x, oa[k]);
      oa[k] = fmaf(hv[1], w2.y, oa[k]);
      ob[k] = fmaf(hv[2], w2.x, ob[k]);
      ob[k] = fmaf(hv[3], w2.y, ob[k]);
    }
  }
#pragma unroll
  for (int s = 1; s <= 2; s <<= 1) {
#pragma unroll
    for (int k = 0; k < QOT_OUT; ++k) {
      oa[k] += __shfl_xor_sync(kFull, oa[k], s);
      ob[k] += __shfl_xor_sync(kFull, ob[k], s);
    }
  }
  const float b2 = t4 < QOT_OUT ? __ldg(prep + kOffB2 + t4) : 0.f;
  oa_out = (t4 == 0 ? oa[0] : t4 == 1 ? oa[1] : oa[2]) + b2;
  ob_out = (t4 == 0 ? ob[0] : t4 == 1 ? ob[1] : ob[2]) + b2;
}

// descriptor of the batch tile T of the launch belongs to (uniform tile count per batch, or prefix search)
// T is absolute (tile0 units); the launch covers tiles [base, base + total)
__device__ __forceinline__ int st_batch_of(const qot_lp_batch_t* __restrict__ bt, int nb, int64_t tpb, int64_t base, int64_t T) {
  if (tpb > 0) return static_cast<int>(min((T - base) / tpb, static_cast<int64_t>(nb - 1)));
  int lo = 0, hi = nb - 1;                 // last b with tile0[b] <= T
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (bt[mid].tile0 <= T) lo = mid; else hi = mid - 1;
  }
  return lo;
}

constexpr int kSubMsg = 16;               // fast path: sources of the LUT row + its self loop

}  // namespace qot
