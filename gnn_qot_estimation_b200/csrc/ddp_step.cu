// Tail of the data-parallel training step in ONE launch: gradient exchange + SGD update.
//
// The reference trains single-process (topological_training/train.py:107-116: loss.backward(); optimizer.step()
// with torch.optim.SGD(lr .1, momentum .9), :66); data parallelism over the GPUs of a box is the new capability
// BASELINE.json's north_star asks for.  The gradient is 17-21 KB (5 291 floats): an all-reduce of that size is pure
// latency, and a library collective costs more than the whole backward kernel once eight processes issue it every
// 0.15 ms.  So the exchange is a ONE-SHOT all-reduce over NVLink peer memory inside the kernel that also applies the
// update:
//   1. every rank copies its flat gradient into its own exchange buffer (memory every peer has mapped: CUDA IPC /
//      torch symmetric memory), slot = step parity;
//   2. flag exchange: rank r stores the step number into word r of every peer's flag row (st.release.sys) and waits
//      until its own row shows the step number from every peer (ld.acquire.sys) -- the only synchronisation;
//   3. every rank reads all W slots over NVLink (L1-bypassing loads), sums them in rank order 0..W-1 -- the same
//      order everywhere, so the replicas stay bit-identical -- scales by 1/W, writes the averaged gradient back to
//      its flat gradient buffer (p.grad views see it, as after a DDP all-reduce);
//   4. torch.optim.SGD's update rule (weight decay, momentum, dampening, nesterov, maximize) on the flat momentum
//      buffer and the parameter tensors (a table of segments), hyper-parameters read from DEVICE memory so that a
//      captured step follows an lr schedule without re-capture.
// Double buffering by step parity makes a trailing barrier unnecessary: a rank can only overwrite slot p at step
// s + 2 after it passed the flag exchange of step s + 1, which every peer enters only after it finished reading
// step s.  World size 1 skips 1-3 (no peers), keeping the fused update.  One CTA: the work is 5 k elements.
#include "common.cuh"

namespace qot {

constexpr int kDdpThreads = 1024;
constexpr int kDdpMaxWorld = 16;
constexpr int kDdpMaxSegs = 256;             // parameter tensors of one model (the reference models have 20 / 15)
constexpr unsigned long long kDdpTimeoutNs = 4000000000ull;   // a peer that never arrives ends the kernel (status), not a hang

// L1-bypassing 16-byte load of a peer's slot (the same addresses are rewritten every second step)
__device__ __forceinline__ float4 ld_peer4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

__global__ void __launch_bounds__(kDdpThreads, 1)
ddp_sgd_step_kernel(float* __restrict__ grad, float* const* __restrict__ peers, int world, int rank, int64_t n, int64_t n_pad,
                    const qot_param_seg_t* __restrict__ segs, int nseg, float* __restrict__ momentum_buf,
                    const qot_sgd_hyper_t* __restrict__ hyper, unsigned long long* __restrict__ state,
                    int32_t* __restrict__ status) {
  const int tid = threadIdx.x;
  const unsigned long long step = state[0] + 1ull;                // 1, 2, 3, ...: the flag value of this step
  __shared__ int timed_out;
  __shared__ long long seg_off[kDdpMaxSegs];
  __shared__ float* seg_ptr[kDdpMaxSegs];
  if (tid == 0) timed_out = 0;
  for (int j = tid; j < nseg; j += kDdpThreads) {
    seg_off[j] = segs[j].offset;
    seg_ptr[j] = segs[j].param;
  }
  __syncthreads();
  if (world > 1) {
    float* mine = peers[rank] + (step & 1ull) * n_pad;
    for (int64_t i = tid; i < n; i += kDdpThreads) mine[i] = grad[i];
    __threadfence_system();
    __syncthreads();
    if (tid < world) {
      unsigned* their_flags = reinterpret_cast<unsigned*>(peers[tid] + 2 * n_pad);
      const unsigned v = static_cast<unsigned>(step);
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(their_flags + rank), "r"(v) : "memory");
      const unsigned* my_flags = reinterpret_cast<const unsigned*>(peers[rank] + 2 * n_pad);
      unsigned long long t0;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
      for (;;) {
        unsigned got;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(got) : "l"(my_flags + tid) : "memory");
        if (static_cast<int>(got - v) >= 0) break;                // peers may already be one step ahead
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > kDdpTimeoutNs) { timed_out = 1; break; }
      }
    }
    __syncthreads();
    if (timed_out) {
      if (tid == 0) atomicOr(status, 1);
      return;                                                     // no update: the replicas would diverge
    }
  }
  // one_minus_dampening: rounded from double on the host, as torch's alpha = 1 - dampening (not 1.0f - float(dampening))
  const float lr = hyper->lr, mom = hyper->momentum, omd = hyper->one_minus_dampening, wd = hyper->weight_decay;
  const bool nesterov = hyper->nesterov != 0, maximize = hyper->maximize != 0;
  const float inv_w = 1.0f / static_cast<float>(world);
  const bool first = mom != 0.f && state[1] == 0ull;             // torch: the first step clones the gradient into the buffer
  // four elements per thread and iteration; the W remote loads of an iteration are all in flight before the first is
  // used (a dependent load-add chain over NVLink would cost one ~1 us round trip per peer and element)
  for (int64_t u = tid; u < n_pad / 4; u += kDdpThreads) {
    const int64_t i0 = 4 * u;
    float gq[4];
    if (world > 1) {
      float4 v[kDdpMaxWorld];
#pragma unroll
      for (int r = 0; r < kDdpMaxWorld; ++r)
        if (r < world) v[r] = ld_peer4(peers[r] + (step & 1ull) * n_pad + i0);
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int r = 0; r < kDdpMaxWorld; ++r)                      // fixed order: rank 0 .. W-1, the same on every rank
        if (r < world) { acc.x += v[r].x; acc.y += v[r].y; acc.z += v[r].z; acc.w += v[r].w; }
      gq[0] = acc.x * inv_w; gq[1] = acc.y * inv_w; gq[2] = acc.z * inv_w; gq[3] = acc.w * inv_w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) gq[j] = i0 + j < n ? grad[i0 + j] : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t i = i0 + j;
      if (i >= n) break;
      float g = gq[j];
      if (world > 1) grad[i] = g;
      // segment of element i (parameters in FlatGradBuffer order)
      int lo = 0, hi = nseg - 1;
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (seg_off[mid] <= i) lo = mid; else hi = mid - 1;
      }
      float* pp = seg_ptr[lo] + (i - seg_off[lo]);
      float p = *pp;
      // torch.optim.SGD (torch/optim/sgd.py, _multi_tensor_sgd), rounding step by step as its foreach kernels do
      if (maximize) g = -g;
      if (wd != 0.f) g = fmaf(wd, p, g);
      if (mom != 0.f) {
        float b = first ? g : fmaf(omd, g, __fmul_rn(momentum_buf[i], mom));
        momentum_buf[i] = b;
        g = nesterov ? fmaf(mom, b, g) : b;
      }
      *pp = fmaf(-lr, g, p);
    }
  }
  __syncthreads();
  if (tid == 0) {
    state[0] = step;
    if (mom != 0.f) state[1] = 1ull;
  }
}

}  // namespace qot

using namespace qot;

extern "C" size_t qot_ddp_exchange_bytes(int64_t n) {
  if (n < 0) return 0;
  const size_t n_pad = (static_cast<size_t>(n) + 63) / 64 * 64;
  return 2 * n_pad * 4 + 4 * 64;                        // two gradient slots + one flag word per peer
}

extern "C" int qot_ddp_sgd_step(float* grad, float* const* peers, int32_t world, int32_t rank, int64_t n,
                                const qot_param_seg_t* segs, int32_t nseg, float* momentum_buf,
                                const qot_sgd_hyper_t* hyper, unsigned long long* state, int32_t* status,
                                void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  QOT_REQUIRE(grad && segs && momentum_buf && hyper && state && status && n > 0 && nseg > 0, "qot_ddp_sgd_step: bad argument");
  QOT_REQUIRE(nseg <= kDdpMaxSegs, "qot_ddp_sgd_step: more than %d parameter tensors", kDdpMaxSegs);
  QOT_REQUIRE(world >= 1 && world <= kDdpMaxWorld && rank >= 0 && rank < world, "qot_ddp_sgd_step: bad world / rank");
  QOT_REQUIRE(world == 1 || peers, "qot_ddp_sgd_step: peers missing");
  const int64_t n_pad = (n + 63) / 64 * 64;
  ddp_sgd_step_kernel<<<1, kDdpThreads, 0, stream>>>(grad, peers, world, rank, n, n_pad, segs, nseg, momentum_buf, hyper,
                                                    state, status);
  QOT_LAUNCH_CHECK();
  return QOT_OK;
}
