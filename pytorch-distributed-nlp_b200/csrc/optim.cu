// Gradient exchange + optimizer in one pass over HBM.
//
// Replaces three things the reference does separately and un-overlapped (SURVEY.md K13-K15):
//   optimizer.zero_grad()            multi-gpu-distributed-cls.py:172   (grads are consumed in place, never re-zeroed)
//   DDP Reducer bucket all-reduce    SP/torch/nn/parallel/distributed.py:1255-1280, reducer.hpp:276-286
//   HF AdamW.step python loop        transformers 4.28.1 optimization.py::AdamW.step (~1600 launches/step)
//
// Each rank owns a contiguous 1/world slice of every bucket: it reads that slice of the bf16 gradients straight
// out of every peer's HBM (NVSwitch peer loads), sums in fp32 in fixed rank order, divides by world (DDP's mean),
// applies the HF AdamW update to its fp32 master weights / moments, and stores the refreshed bf16 shadow weights
// into every peer's weight buffer (NVSwitch peer stores).  world == 1 degenerates to a fused multi-tensor AdamW.
#include "common.cuh"
#include "../../include/b2_ddp_bert.h"

namespace b2 {

constexpr int MAX_WORLD = 8;

struct ReduceAdamWParams {
  const __nv_bfloat16* grads[MAX_WORLD];
  __nv_bfloat16* shadow[MAX_WORLD];
  int world;
  float* master; float* m; float* v;
  const uint8_t* decay;
  long long begin, end;  // element range, multiples of 8
  // scalars pre-rounded on the host exactly as torch rounds the python doubles HF AdamW passes to its ATen ops
  double lr_d, beta1_d, beta2_d;
  float lr, beta1, beta2, one_minus_beta1, one_minus_beta2, eps, lr_wd;
  int correct_bias, has_wd;
  const long long* step_counter;
  const float* grad_scale;   // optional device scalar (GradScaler): gradients are divided by it
  const float* found_inf;    // optional device scalar (GradScaler): non-zero skips the update
  const uint8_t* skip;       // optional per-vector flags: already updated by the fused wgrad epilogue
};

__global__ void __launch_bounds__(256) reduce_adamw_kernel(const ReduceAdamWParams p) {
  pdl_wait();               // PDL: predecessors complete + visible before any global access
  pdl_launch_dependents();  // let the next kernel in the stream begin launching
  if (p.found_inf != nullptr && *p.found_inf != 0.f) return;   // GradScaler saw inf/nan: this step is skipped
  // HF AdamW bias correction: step_size = lr * sqrt(1 - b2^t) / (1 - b1^t), t = steps taken including this one
  const long long t = *p.step_counter + 1;
  float step_size = p.lr;
  if (p.correct_bias) {
    const double bc1 = 1.0 - pow(p.beta1_d, (double)t);
    const double bc2 = 1.0 - pow(p.beta2_d, (double)t);
    step_size = (float)(p.lr_d * sqrt(bc2) / bc1);
  }
  // mean over ranks; with a GradScaler also the unscale (a power of two: exact)
  const float inv_world = (p.grad_scale != nullptr ? 1.0f / *p.grad_scale : 1.0f) / (float)p.world;
  const long long nvec = (p.end - p.begin) >> 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec;
       i += (long long)gridDim.x * blockDim.x) {
    const long long e = p.begin + (i << 3);
    if (p.skip != nullptr && p.skip[e >> 3]) continue;
    float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int r = 0; r < MAX_WORLD; ++r) {
      if (r < p.world) {
        // peer-mapped pointer: plain 16-byte global load; the address aperture routes it over NVLink
        const uint4 q = *reinterpret_cast<const uint4*>(p.grads[r] + e);
        g[0] += bf16_lo(q.x); g[1] += bf16_hi(q.x); g[2] += bf16_lo(q.y); g[3] += bf16_hi(q.y);
        g[4] += bf16_lo(q.z); g[5] += bf16_hi(q.z); g[6] += bf16_lo(q.w); g[7] += bf16_hi(q.w);
      }
    }
    const bool decay = p.has_wd && p.decay[e >> 3];
    float4 w0 = *reinterpret_cast<const float4*>(p.master + e), w1 = *reinterpret_cast<const float4*>(p.master + e + 4);
    float4 m0 = *reinterpret_cast<const float4*>(p.m + e), m1 = *reinterpret_cast<const float4*>(p.m + e + 4);
    float4 v0 = *reinterpret_cast<const float4*>(p.v + e), v1 = *reinterpret_cast<const float4*>(p.v + e + 4);
    float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
    float mm[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
    float vv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float gk = g[k] * inv_world;
      mm[k] = mm[k] * p.beta1 + gk * p.one_minus_beta1;
      vv[k] = vv[k] * p.beta2 + gk * gk * p.one_minus_beta2;
      const float denom = sqrtf(vv[k]) + p.eps;
      w[k] = w[k] - step_size * (mm[k] / denom);
      if (decay) w[k] = w[k] - p.lr_wd * w[k];
    }
    *reinterpret_cast<float4*>(p.master + e) = make_float4(w[0], w[1], w[2], w[3]);
    *reinterpret_cast<float4*>(p.master + e + 4) = make_float4(w[4], w[5], w[6], w[7]);
    *reinterpret_cast<float4*>(p.m + e) = make_float4(mm[0], mm[1], mm[2], mm[3]);
    *reinterpret_cast<float4*>(p.m + e + 4) = make_float4(mm[4], mm[5], mm[6], mm[7]);
    *reinterpret_cast<float4*>(p.v + e) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    *reinterpret_cast<float4*>(p.v + e + 4) = make_float4(vv[4], vv[5], vv[6], vv[7]);
    uint4 o;
    o.x = pack_bf16(w[0], w[1]); o.y = pack_bf16(w[2], w[3]);
    o.z = pack_bf16(w[4], w[5]); o.w = pack_bf16(w[6], w[7]);
#pragma unroll
    for (int r = 0; r < MAX_WORLD; ++r)
      if (r < p.world && p.shadow[r] != nullptr) *reinterpret_cast<uint4*>(p.shadow[r] + e) = o;
  }
}

// ---- single-GPU background form ------------------------------------------------------------------------------------
// Measured (B2_DEBUG_SKIP_ADAMW): on one GPU the 0.49 ms of optimizer kernels are exposed almost in full, although they
// run on their own stream under the backward pass -- a 256-thread x 64-register block cannot become resident on an SM
// whose 64 K registers are held by a 640-thread x 96-register GEMM CTA (61 440), so the update only ever runs in the
// gaps between GEMM kernels.  This variant is shaped to fit BESIDE such a CTA: 128 threads x 32 registers = the 4 096
// registers that are left, no shared memory, and the same shared-memory carve-out preference as the GEMM kernels
// (an SM is not re-partitioned while it has resident CTAs).  Blocks are short-lived (8 vectors of 4 elements per
// thread) so they never hold an SM back from a kernel that needs all of it (the attention kernels).  Same arithmetic,
// statement for statement, as reduce_adamw_kernel with world == 1; the bias-corrected step size is computed once per
// step by adamw_prepare_kernel (double pow, as the host would) instead of in every block.
// Measured (tools/coresidency_probe.py: a GEMM loop on one stream, the update of all 102 M parameters on another):
// the blocks do become co-resident, but one 128-thread block per SM keeps only ~7 KB in flight: 27 % of the update
// hides under the GEMMs (the 256-thread form: none -- it even costs 20 % more than running the two back to back);
// in the training step +1.2 % (7 987 -> 8 085 samples/s).  Asking the L2 for the operands of a later block first
// (cp.async.bulk.prefetch.L2, no registers held) was tried and measured worse (19 % hidden): the co-resident blocks are
// bound by the latency of their own dependent load -> sqrt -> divide -> store chain, not by HBM queue depth.
struct SlimParams {
  const __nv_bfloat16* grads; __nv_bfloat16* shadow;
  float* master; float* m; float* v;
  const uint8_t* decay;
  long long begin, nvec4;
  float beta1, beta2, one_minus_beta1, one_minus_beta2, eps, lr_wd;
  int has_wd;
  const float* step_size;
};
constexpr int kSlimThreads = 128, kSlimIters = 8;
template <int DUMMY>
__global__ void __launch_bounds__(DUMMY > 0 ? kSlimThreads : 0) __maxnreg__(DUMMY > 0 ? 32 : 24)
adamw_slim_kernel(const SlimParams p) {
  pdl_wait();
  pdl_launch_dependents();
  const float step_size = *p.step_size;
  long long i = (long long)blockIdx.x * (kSlimThreads * kSlimIters) + threadIdx.x;
#pragma unroll 1
  for (int it = 0; it < kSlimIters; ++it, i += kSlimThreads) {
    if (i >= p.nvec4) break;
    const long long e = p.begin + (i << 2);
    const uint2 q = *reinterpret_cast<const uint2*>(p.grads + e);
    float4 w = *reinterpret_cast<const float4*>(p.master + e);
    float4 mm = *reinterpret_cast<const float4*>(p.m + e);
    float4 vv = *reinterpret_cast<const float4*>(p.v + e);
    const bool decay = p.has_wd && p.decay[e >> 3];
    const float g0 = bf16_lo(q.x), g1 = bf16_hi(q.x), g2 = bf16_lo(q.y), g3 = bf16_hi(q.y);
    mm.x = mm.x * p.beta1 + g0 * p.one_minus_beta1; vv.x = vv.x * p.beta2 + g0 * g0 * p.one_minus_beta2;
    mm.y = mm.y * p.beta1 + g1 * p.one_minus_beta1; vv.y = vv.y * p.beta2 + g1 * g1 * p.one_minus_beta2;
    mm.z = mm.z * p.beta1 + g2 * p.one_minus_beta1; vv.z = vv.z * p.beta2 + g2 * g2 * p.one_minus_beta2;
    mm.w = mm.w * p.beta1 + g3 * p.one_minus_beta1; vv.w = vv.w * p.beta2 + g3 * g3 * p.one_minus_beta2;
    w.x = w.x - step_size * (mm.x / (sqrtf(vv.x) + p.eps));
    w.y = w.y - step_size * (mm.y / (sqrtf(vv.y) + p.eps));
    w.z = w.z - step_size * (mm.z / (sqrtf(vv.z) + p.eps));
    w.w = w.w - step_size * (mm.w / (sqrtf(vv.w) + p.eps));
    if (decay) {
      w.x = w.x - p.lr_wd * w.x; w.y = w.y - p.lr_wd * w.y; w.z = w.z - p.lr_wd * w.z; w.w = w.w - p.lr_wd * w.w;
    }
    *reinterpret_cast<float4*>(p.master + e) = w;
    *reinterpret_cast<float4*>(p.m + e) = mm;
    *reinterpret_cast<float4*>(p.v + e) = vv;
    uint2 o;
    o.x = pack_bf16(w.x, w.y);
    o.y = pack_bf16(w.z, w.w);
    *reinterpret_cast<uint2*>(p.shadow + e) = o;
  }
}

// HF AdamW bias correction for the NEXT update: step_size = lr * sqrt(1 - b2^t) / (1 - b1^t), t = *step + 1
__global__ void adamw_prepare_kernel(double lr, double beta1, double beta2, int correct_bias, const long long* step,
                                     float* step_size) {
  pdl_wait();
  pdl_launch_dependents();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double ss = lr;
    if (correct_bias) {
      const long long t = *step + 1;
      ss = lr * sqrt(1.0 - pow(beta2, (double)t)) / (1.0 - pow(beta1, (double)t));
    }
    *step_size = (float)ss;
  }
}

__global__ void step_advance_kernel(long long* step, unsigned long long* rng, const float* found_inf) {
  pdl_wait();               // PDL: predecessors complete + visible before any global access
  pdl_launch_dependents();  // let the next kernel in the stream begin launching
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (step && !(found_inf != nullptr && *found_inf != 0.f)) *step += 1;
    if (rng) rng[1] += 1;
  }
}
__global__ void rng_seed_kernel(unsigned long long* rng, unsigned long long seed, unsigned long long step) {
  pdl_wait();               // PDL: predecessors complete + visible before any global access
  pdl_launch_dependents();  // let the next kernel in the stream begin launching
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    rng[0] = seed;
    rng[1] = step;
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n) {
  pdl_wait();               // PDL: predecessors complete + visible before any global access
  pdl_launch_dependents();  // let the next kernel in the stream begin launching
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i + 8 <= n) {
    const float4 a = *reinterpret_cast<const float4*>(src + i), b = *reinterpret_cast<const float4*>(src + i + 4);
    uint4 o;
    o.x = pack_bf16(a.x, a.y); o.y = pack_bf16(a.z, a.w); o.z = pack_bf16(b.x, b.y); o.w = pack_bf16(b.z, b.w);
    stg16(dst + i, o);
  } else {
    for (long long k = i; k < n; ++k) dst[k] = __float2bfloat16_rn(src[k]);
  }
}
__global__ void cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, long long n) {
  pdl_wait();               // PDL: predecessors complete + visible before any global access
  pdl_launch_dependents();  // let the next kernel in the stream begin launching
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __bfloat162float(src[i]);
}

// ---- gradient accumulation (no_sync() micro-batches) ----------------------------------------------------------------
// Folds one micro-batch's bf16 gradient into the fp32 accumulator: ADD acc += scale * g, FINISH g = bf16(acc + scale *
// g) and acc = 0.  Launched per bucket under the backward pass (optimizer stream / DDP side stream), so it has the shape
// of adamw_slim_kernel: 128 threads, at most 32 registers, no shared memory, short-lived blocks; 16-byte accesses
// (8 elements per thread and iteration).  10 B per parameter for ADD, 12 B for FINISH.
struct AccumParams {
  float* acc; __nv_bfloat16* grads;
  long long begin, nvec8;
  float scale;
};
constexpr int kAccumThreads = 128, kAccumIters = 4;
template <int MODE>
__global__ void __launch_bounds__(MODE >= 0 ? kAccumThreads : 0) __maxnreg__(MODE >= 0 ? 32 : 24)
grad_accumulate_kernel(const AccumParams p) {
  pdl_wait();
  pdl_launch_dependents();
  long long i = (long long)blockIdx.x * (kAccumThreads * kAccumIters) + threadIdx.x;
#pragma unroll 1
  for (int it = 0; it < kAccumIters; ++it, i += kAccumThreads) {
    if (i >= p.nvec8) break;
    const long long e = p.begin + (i << 3);
    const uint4 q = *reinterpret_cast<const uint4*>(p.grads + e);
    float4 a0 = *reinterpret_cast<const float4*>(p.acc + e), a1 = *reinterpret_cast<const float4*>(p.acc + e + 4);
    a0.x += p.scale * bf16_lo(q.x); a0.y += p.scale * bf16_hi(q.x);
    a0.z += p.scale * bf16_lo(q.y); a0.w += p.scale * bf16_hi(q.y);
    a1.x += p.scale * bf16_lo(q.z); a1.y += p.scale * bf16_hi(q.z);
    a1.z += p.scale * bf16_lo(q.w); a1.w += p.scale * bf16_hi(q.w);
    if (MODE == B2_ACCUM_ADD) {
      *reinterpret_cast<float4*>(p.acc + e) = a0;
      *reinterpret_cast<float4*>(p.acc + e + 4) = a1;
    } else {
      uint4 o;
      o.x = pack_bf16(a0.x, a0.y); o.y = pack_bf16(a0.z, a0.w);
      o.z = pack_bf16(a1.x, a1.y); o.w = pack_bf16(a1.z, a1.w);
      *reinterpret_cast<uint4*>(p.grads + e) = o;
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(p.acc + e) = z;
      *reinterpret_cast<float4*>(p.acc + e + 4) = z;
    }
  }
}

// segments [n][3] = {src offset, dst offset, count}: dst(bf16) <- src(fp32); src <- 0.  grid = (ceil(max_count/256), n)
__global__ void accum_finish_kernel(float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                    const long long* __restrict__ seg) {
  pdl_wait();
  pdl_launch_dependents();
  const long long so = seg[blockIdx.y * 3], d0 = seg[blockIdx.y * 3 + 1], cnt = seg[blockIdx.y * 3 + 2];
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cnt) {
    dst[d0 + i] = __float2bfloat16_rn(src[so + i]);
    src[so + i] = 0.f;
  }
}

}  // namespace b2

using namespace b2;

extern "C" int32_t b2_accum_finish(float* src, void* dst, const int64_t* segments, int64_t n_segments,
                                   int64_t max_count, void* stream_) {
  B2_REQUIRE(src && dst && segments && n_segments > 0 && max_count > 0, "accum_finish: bad args");
  dim3 grid((unsigned)((max_count + 255) / 256), (unsigned)n_segments);
  B2_LAUNCH(accum_finish_kernel, grid, 256, 0, stream_, src, (__nv_bfloat16*)dst, (const long long*)segments);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_bucket_reduce_adamw(const void* const* peer_grads, void* const* peer_shadow, int32_t world,
                                          int32_t rank, float* master, float* exp_avg, float* exp_avg_sq,
                                          const uint8_t* decay_flags, int64_t begin, int64_t end,
                                          const b2_adamw_hparams_t* hp, const int64_t* step_counter, void* stream_) {
  B2_REQUIRE(peer_grads && peer_shadow && master && exp_avg && exp_avg_sq && decay_flags && hp && step_counter,
             "bucket_reduce_adamw: null pointer");
  B2_REQUIRE(world >= 1 && world <= MAX_WORLD && rank >= 0 && rank < world, "bucket_reduce_adamw: world=%d rank=%d",
             world, rank);
  B2_REQUIRE(begin >= 0 && end >= begin && begin % 8 == 0 && end % 8 == 0,
             "bucket_reduce_adamw: slice [%lld,%lld) must be 8-element aligned", (long long)begin, (long long)end);
  if (end == begin) return 0;
  ReduceAdamWParams p;
  for (int r = 0; r < MAX_WORLD; ++r) {
    p.grads[r] = r < world ? (const __nv_bfloat16*)peer_grads[r] : nullptr;
    p.shadow[r] = r < world ? (__nv_bfloat16*)peer_shadow[r] : nullptr;
    // a NULL shadow entry = that peer's copy is delivered some other way (copy-engine all-gather)
    if (r < world) B2_REQUIRE(p.grads[r] && (p.shadow[r] || r != rank), "bucket_reduce_adamw: null peer pointer for rank %d", r);
  }
  p.world = world;
  p.master = master; p.m = exp_avg; p.v = exp_avg_sq; p.decay = decay_flags;
  p.begin = begin; p.end = end;
  p.lr_d = hp->lr; p.beta1_d = hp->beta1; p.beta2_d = hp->beta2;
  p.lr = (float)hp->lr; p.beta1 = (float)hp->beta1; p.beta2 = (float)hp->beta2;
  p.one_minus_beta1 = (float)(1.0 - hp->beta1); p.one_minus_beta2 = (float)(1.0 - hp->beta2);
  p.eps = (float)hp->eps; p.lr_wd = (float)(hp->lr * hp->weight_decay);
  p.correct_bias = hp->correct_bias; p.has_wd = hp->weight_decay > 0.0 ? 1 : 0;
  p.step_counter = (const long long*)step_counter;
  p.grad_scale = hp->grad_scale;
  p.found_inf = hp->found_inf;
  p.skip = hp->skip_flags;
  const long long nvec = (end - begin) >> 3;
  long long blocks = (nvec + 255) / 256;
  const long long cap = 148 * 8;
  if (blocks > cap) blocks = cap;
  B2_LAUNCH(reduce_adamw_kernel, (unsigned)blocks, 256, 0, (cudaStream_t)stream_, p);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_adamw_prepare(const b2_adamw_hparams_t* hp, const int64_t* step_counter, float* step_size,
                                    void* stream_) {
  B2_REQUIRE(hp && step_counter && step_size, "adamw_prepare: null pointer");
  B2_LAUNCH(adamw_prepare_kernel, 1, 32, 0, (cudaStream_t)stream_, hp->lr, hp->beta1, hp->beta2, hp->correct_bias,
            (const long long*)step_counter, step_size);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_adamw_background(const void* grads, void* shadow, float* master, float* exp_avg,
                                       float* exp_avg_sq, const uint8_t* decay_flags, int64_t begin, int64_t end,
                                       const b2_adamw_hparams_t* hp, const float* step_size, void* stream_) {
  B2_REQUIRE(grads && shadow && master && exp_avg && exp_avg_sq && decay_flags && hp && step_size,
             "adamw_background: null pointer");
  B2_REQUIRE(begin >= 0 && end >= begin && begin % 8 == 0 && end % 8 == 0,
             "adamw_background: slice [%lld,%lld) must be 8-element aligned", (long long)begin, (long long)end);
  B2_REQUIRE(hp->grad_scale == nullptr && hp->found_inf == nullptr && hp->skip_flags == nullptr,
             "adamw_background: GradScaler state / skip flags are handled by b2_bucket_reduce_adamw");
  if (end == begin) return 0;
  static bool attr = false;
  if (!attr) {   // same shared-memory carve-out as the GEMM CTAs it is meant to run beside
    B2_CUDA(cudaFuncSetAttribute(adamw_slim_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared));
    attr = true;
  }
  SlimParams p;
  p.grads = (const __nv_bfloat16*)grads; p.shadow = (__nv_bfloat16*)shadow;
  p.master = master; p.m = exp_avg; p.v = exp_avg_sq; p.decay = decay_flags;
  p.begin = begin; p.nvec4 = (end - begin) >> 2;
  p.beta1 = (float)hp->beta1; p.beta2 = (float)hp->beta2;
  p.one_minus_beta1 = (float)(1.0 - hp->beta1); p.one_minus_beta2 = (float)(1.0 - hp->beta2);
  p.eps = (float)hp->eps; p.lr_wd = (float)(hp->lr * hp->weight_decay);
  p.has_wd = hp->weight_decay > 0.0 ? 1 : 0;
  p.step_size = step_size;
  const long long per_block = (long long)kSlimThreads * kSlimIters;
  const long long blocks = (p.nvec4 + per_block - 1) / per_block;
  B2_LAUNCH(adamw_slim_kernel<1>, (unsigned)blocks, kSlimThreads, 0, (cudaStream_t)stream_, p);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_grad_accumulate(float* acc, void* grads, int64_t begin, int64_t end, float scale, int32_t mode,
                                      void* stream_) {
  B2_REQUIRE(acc && grads, "grad_accumulate: null pointer");
  B2_REQUIRE(begin >= 0 && end >= begin && begin % 8 == 0 && end % 8 == 0,
             "grad_accumulate: range [%lld,%lld) must be 8-element aligned", (long long)begin, (long long)end);
  B2_REQUIRE(mode == B2_ACCUM_ADD || mode == B2_ACCUM_FINISH, "grad_accumulate: mode %d", mode);
  if (end == begin) return 0;
  static bool attr = false;
  if (!attr) {   // same shared-memory carve-out as the GEMM CTAs it runs beside (see adamw_slim_kernel)
    B2_CUDA(cudaFuncSetAttribute(grad_accumulate_kernel<B2_ACCUM_ADD>,
                                 cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    B2_CUDA(cudaFuncSetAttribute(grad_accumulate_kernel<B2_ACCUM_FINISH>,
                                 cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr = true;
  }
  AccumParams p;
  p.acc = acc; p.grads = (__nv_bfloat16*)grads;
  p.begin = begin; p.nvec8 = (end - begin) >> 3;
  p.scale = scale;
  const long long per_block = (long long)kAccumThreads * kAccumIters;
  const long long blocks = (p.nvec8 + per_block - 1) / per_block;
  if (mode == B2_ACCUM_ADD)
    B2_LAUNCH(grad_accumulate_kernel<B2_ACCUM_ADD>, (unsigned)blocks, kAccumThreads, 0, (cudaStream_t)stream_, p);
  else
    B2_LAUNCH(grad_accumulate_kernel<B2_ACCUM_FINISH>, (unsigned)blocks, kAccumThreads, 0, (cudaStream_t)stream_, p);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_step_advance(int64_t* step_counter, void* rng_state, const float* found_inf, void* stream_) {
  B2_LAUNCH(step_advance_kernel, 1, 32, 0, (cudaStream_t)stream_, (long long*)step_counter,
            (unsigned long long*)rng_state, found_inf);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_rng_seed(void* rng_state, uint64_t seed, uint64_t step, void* stream_) {
  B2_REQUIRE(rng_state, "rng_seed: null pointer");
  B2_LAUNCH(rng_seed_kernel, 1, 32, 0, (cudaStream_t)stream_, (unsigned long long*)rng_state, seed, step);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream_) {
  B2_REQUIRE(src && dst && n >= 0, "cast_f32_to_bf16: bad args");
  B2_REQUIRE(((uintptr_t)src % 16 == 0) && ((uintptr_t)dst % 16 == 0), "cast_f32_to_bf16: 16-byte alignment required");
  if (n == 0) return 0;
  const long long nv = (n + 7) / 8;
  B2_LAUNCH(cast_f32_bf16_kernel, (unsigned)((nv + 255) / 256), 256, 0, (cudaStream_t)stream_, src, (__nv_bfloat16*)dst, n);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_cast_bf16_to_f32(const void* src, float* dst, int64_t n, void* stream_) {
  B2_REQUIRE(src && dst && n >= 0, "cast_bf16_to_f32: bad args");
  if (n == 0) return 0;
  B2_LAUNCH(cast_bf16_f32_kernel, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream_, (const __nv_bfloat16*)src, dst,
                                                                                       n);
  B2_CUDA(cudaGetLastError());
  count_launches(1);
  return 0;
}

extern "C" int32_t b2_zero(void* dst, int64_t bytes, void* stream_) {
  B2_REQUIRE(dst && bytes >= 0, "zero: bad args");
  if (bytes == 0) return 0;
  B2_CUDA(cudaMemsetAsync(dst, 0, (size_t)bytes, (cudaStream_t)stream_));
  return 0;
}

extern "C" int32_t b2_copy_async(void* dst, const void* src, int64_t bytes, void* stream_) {
  B2_REQUIRE(dst && src && bytes >= 0, "copy_async: bad args");
  if (bytes == 0) return 0;
  // device-to-device: between a local buffer and an IPC-mapped peer buffer this is a copy-engine transfer over
  // NVLink that runs beside the SM kernels of other streams (a memcpy node when captured in a graph)
  B2_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream_));
  return 0;
}
