// Flat-arena optimizer + collective kernels (sm_100a, NVLink 5 / NVSwitch peer memory).
//
// Every rank maps every peer's *symmetric arena* (W | G | U | R | H regions at identical byte offsets) and a
// small *signal pad* into its own address space (csrc/peer_arena.cpp).  The kernels below therefore issue
// plain ld/st (or multimem.* when a multicast mapping exists) on peer pointers — no NCCL/MPI call is on the
// path.  What the reference does in three separate stages per tensor
//     Barrier → ncclAllReduce(vels→vels2) → one elementwise update kernel per tensor
// (theanompi/lib/exchanger.py:120-134, exchanger_strategy.py:121-127, opt.py:181-268) is ONE launch here:
//     flag barrier → read all peers' gradients → average → weight-decay/momentum/lr update → bf16 shadow
//     [→ push the updated slice to the peers] → flag barrier.
//
//   sgd_flat            k = 1 instance (no peers): fused momentum-SGD over a block range
//   fused_oneshot_sgd   every rank reduces the whole range itself (latency-optimal, small buckets)
//   fused_twoshot_sgd   reduce-scatter → update owned slice → push updated weights to all peers (bandwidth-optimal)
//   fused_nvls_sgd      same with multimem.ld_reduce / multimem.st (reduction + broadcast inside the NVSwitch)
//   allreduce_*         plain sum/avg into a destination region (classic cdd vels→vels2, 'avg' weight averaging)
//   easgd_elastic       d = α(w − c); w −= d; c += d   on the center's memory over NVLink   (exchanger.py:188-211)
//   gosgd_*             push / merge / pull-merge of weights with push-sum weights α     (exchanger.py:450-462)
//   K1..K5 of the reference (float2half/half2float, sumfloats/sumhalfs, vecadd/vecaddhalf) for the legacy strategies.
#include "common.cuh"
#include "api.h"

namespace tmpi {

constexpr int kThreads = 256;            // one float4 per thread per 1024-element arena block

// ------------------------------------------------------------------ memory helpers
__device__ __forceinline__ float4 ld_sys_f4(const float* p) {
  float4 v;
  asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint2 ld_sys_u2(const void* p) {
  uint2 v;
  asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_f4(float* p, float4 v) {
  asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_u2(void* p, uint2 v) {
  asm volatile("st.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ float4 mc_ld_reduce_f4(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ uint2 mc_ld_reduce_bf16x4(const void* mc) {
  uint2 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v2.bf16x2 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void mc_st_f4(float* mc, float4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void mc_st_u2(void* mc, uint2 v) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1, %2};" ::"l"(mc), "f"(__uint_as_float(v.x)), "f"(__uint_as_float(v.y)) : "memory");
}
__device__ __forceinline__ uint2 pack_bf16x4(float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 r; r.x = *reinterpret_cast<uint32_t*>(&a); r.y = *reinterpret_cast<uint32_t*>(&b); return r;
}
__device__ __forceinline__ float4 unpack_bf16x4(uint2 u) {
  float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u.x)), b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

template <typename T> __device__ __forceinline__ T* region(const CommCtx& c, int p, long long off) {
  return reinterpret_cast<T*>(reinterpret_cast<char*>(c.arena[p]) + off);
}

// ------------------------------------------------------------------ cross-rank per-block flag barrier
// Block b of every rank increments slot [b][my rank] on every peer (red.release.sys) and spins until its own
// slots [b][p] reach the block's epoch (ld.acquire.sys).  Epochs live in device memory, so the same captured
// CUDA graph can be replayed.  Bounded spin: a protocol bug traps instead of hanging the GPU.
__device__ __forceinline__ void block_barrier(const CommCtx& c) {
  __syncthreads();
  uint32_t* ep = c.epoch + blockIdx.x;
  const uint32_t target = *ep + 1u;
  if ((int)threadIdx.x < c.world) {
    uint32_t* remote = c.sig[threadIdx.x] + (size_t)blockIdx.x * kMaxRanks + c.rank;
    asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(remote) : "memory");
    const uint32_t* mine = c.sig[c.rank] + (size_t)blockIdx.x * kMaxRanks + threadIdx.x;
    uint32_t v;
    long long t0 = clock64();
    while (true) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if ((int)(v - target) >= 0) break;
      if (clock64() - t0 > c.spin_limit) { __trap(); }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *ep = target;
}

// ------------------------------------------------------------------ the SGD math (one float4)
struct Hyper { float lr, mu, inv_k; int nesterov; };

__device__ __forceinline__ void sgd4(float4& w, float4& u, const float4& gsum, const Hyper& h, float lrm, float wd) {
  const float lr = h.lr * lrm;
#define TMPI_SGD1(W, U, G)                                   \
  {                                                          \
    const float ge = G * h.inv_k + wd * W;                   \
    U = h.mu * U + ge;                                       \
    W -= lr * (h.nesterov ? (ge + h.mu * U) : U);            \
  }
  TMPI_SGD1(w.x, u.x, gsum.x) TMPI_SGD1(w.y, u.y, gsum.y) TMPI_SGD1(w.z, u.z, gsum.z) TMPI_SGD1(w.w, u.w, gsum.w)
#undef TMPI_SGD1
}

// ============================================================================ k = 1: local fused SGD
// filter: 0 all groups, 1 only non-exchanged (BN) groups, 2 only exchanged groups
__global__ void __launch_bounds__(kThreads) sgd_flat_kernel(float* __restrict__ W, const float* __restrict__ G, float* __restrict__ U,
                                                            __nv_bfloat16* __restrict__ H, const uint8_t* __restrict__ block_group,
                                                            GroupTable tab, const float* __restrict__ lr_ptr, float mu, int nesterov,
                                                            float inv_k, long long blk_lo, long long blk_hi, int filter) {
  const Hyper h{*lr_ptr, mu, inv_k, nesterov};
  for (long long b = blk_lo + blockIdx.x; b < blk_hi; b += gridDim.x) {
    const int g = block_group[b];
    if ((filter == 1 && tab.exch[g]) || (filter == 2 && !tab.exch[g])) continue;
    const long long i = b * kArenaBlock + threadIdx.x * 4;
    float4 w = *reinterpret_cast<const float4*>(W + i);
    float4 u = *reinterpret_cast<const float4*>(U + i);
    const float4 gg = *reinterpret_cast<const float4*>(G + i);
    sgd4(w, u, gg, h, tab.lr_mult[g], tab.wd[g]);
    *reinterpret_cast<float4*>(W + i) = w;
    *reinterpret_cast<float4*>(U + i) = u;
    if (H) *reinterpret_cast<uint2*>(H + i) = pack_bf16x4(w);
  }
}

void sgd_flat(void* W, const void* G, void* U, void* H, const void* block_group, const GroupTable& tab, const void* lr_ptr, float mu,
              int nesterov, float inv_k, long long lo, long long hi, int filter, cudaStream_t st) {
  if (lo % kArenaBlock || hi % kArenaBlock) throw std::runtime_error("sgd_flat: range must be block aligned");
  const long long nb = (hi - lo) / kArenaBlock;
  if (nb <= 0) return;
  int grid = (int)std::min<long long>(nb, (long long)sm_count() * 8);
  sgd_flat_kernel<<<grid, kThreads, 0, st>>>((float*)W, (const float*)G, (float*)U, (__nv_bfloat16*)H, (const uint8_t*)block_group, tab,
                                             (const float*)lr_ptr, mu, nesterov, inv_k, lo / kArenaBlock, hi / kArenaBlock, filter);
  count_launch(); TMPI_CHECK_LAUNCH("sgd_flat"); ::tmpi::check_capture(st, "sgd_flat");
}

// ============================================================================ flat Adam (Wide-ResNet's optimizer, ref keras_model_zoo/wresnet.py:159)
// ge = inv_k g + wd w;  m = b1 m + (1 - b1) ge;  v = b2 v + (1 - b2) ge^2;  w -= lr * (m / (1 - b1^t)) / (sqrt(v / (1 - b2^t)) + eps),
// t read from a device counter (the captured CUDA graph keeps counting), lr from device memory, bf16 shadow refreshed.
struct AdamHyper { float lr, inv_k, b1, b2, eps, c1, c2; };

__device__ __forceinline__ AdamHyper adam_hyper(const float* lr_ptr, const unsigned long long* step, float inv_k, float b1, float b2,
                                                float eps) {
  const float t = (float)(*step + 1ull);
  return AdamHyper{*lr_ptr, inv_k, b1, b2, eps, 1.f / (1.f - __powf(b1, t)), 1.f / (1.f - __powf(b2, t))};
}

// __fmul_rn keeps g * inv_k out of FMA contraction: with inv_k = 1 the update rounds exactly as  g + wd * w  does
__device__ __forceinline__ void adam4(float4& w, float4& m, float4& v, const float4& gsum, const AdamHyper& h, float lrm, float wd) {
  const float lr = h.lr * lrm;
#define TMPI_ADAM1(Wc, Mc, Vc, Gc)                                    \
  {                                                                  \
    const float ge = __fmul_rn(Gc, h.inv_k) + wd * Wc;               \
    Mc = h.b1 * Mc + (1.f - h.b1) * ge;                              \
    Vc = h.b2 * Vc + (1.f - h.b2) * ge * ge;                         \
    Wc -= lr * (Mc * h.c1) / (sqrtf(Vc * h.c2) + h.eps);             \
  }
  TMPI_ADAM1(w.x, m.x, v.x, gsum.x) TMPI_ADAM1(w.y, m.y, v.y, gsum.y) TMPI_ADAM1(w.z, m.z, v.z, gsum.z) TMPI_ADAM1(w.w, m.w, v.w, gsum.w)
#undef TMPI_ADAM1
}

// filter: 0 all groups, 1 only non-exchanged (BN) groups, 2 only exchanged groups (as sgd_flat)
__global__ void __launch_bounds__(kThreads) adam_flat_kernel(float* __restrict__ W, const float* __restrict__ G, float* __restrict__ M,
                                                             float* __restrict__ V, __nv_bfloat16* __restrict__ H,
                                                             const uint8_t* __restrict__ block_group, GroupTable tab,
                                                             const float* __restrict__ lr_ptr, const unsigned long long* __restrict__ step,
                                                             float b1, float b2, float eps, float inv_k, long long blk_lo, long long blk_hi,
                                                             int filter) {
  const AdamHyper h = adam_hyper(lr_ptr, step, inv_k, b1, b2, eps);
  for (long long b = blk_lo + blockIdx.x; b < blk_hi; b += gridDim.x) {
    const int g = block_group[b];
    if ((filter == 1 && tab.exch[g]) || (filter == 2 && !tab.exch[g])) continue;
    const long long i = b * kArenaBlock + threadIdx.x * 4;
    float4 w = *reinterpret_cast<const float4*>(W + i), m = *reinterpret_cast<const float4*>(M + i), v = *reinterpret_cast<const float4*>(V + i);
    const float4 gg = *reinterpret_cast<const float4*>(G + i);
    adam4(w, m, v, gg, h, tab.lr_mult[g], tab.wd[g]);
    *reinterpret_cast<float4*>(W + i) = w;
    *reinterpret_cast<float4*>(M + i) = m;
    *reinterpret_cast<float4*>(V + i) = v;
    if (H) *reinterpret_cast<uint2*>(H + i) = pack_bf16x4(w);
  }
}
__global__ void adam_advance_kernel(unsigned long long* step) { if (threadIdx.x == 0 && blockIdx.x == 0) *step += 1ull; }

void adam_advance(void* step, cudaStream_t st) {
  adam_advance_kernel<<<1, 32, 0, st>>>((unsigned long long*)step);
  count_launch(); TMPI_CHECK_LAUNCH("adam_advance"); ::tmpi::check_capture(st, "adam_advance");
}

void adam_flat(void* W, const void* G, void* M, void* V, void* H, const void* block_group, const GroupTable& tab, const void* lr_ptr, void* step,
               float b1, float b2, float eps, long long lo, long long hi, float inv_k, int filter, int advance, cudaStream_t st) {
  if (lo % kArenaBlock || hi % kArenaBlock) throw std::runtime_error("adam_flat: range must be block aligned");
  const long long nb = (hi - lo) / kArenaBlock;
  if (nb > 0) {
    int grid = (int)std::min<long long>(nb, (long long)sm_count() * 8);
    adam_flat_kernel<<<grid, kThreads, 0, st>>>((float*)W, (const float*)G, (float*)M, (float*)V, (__nv_bfloat16*)H, (const uint8_t*)block_group,
                                                tab, (const float*)lr_ptr, (const unsigned long long*)step, b1, b2, eps, inv_k, lo / kArenaBlock,
                                                hi / kArenaBlock, filter);
    count_launch(); TMPI_CHECK_LAUNCH("adam_flat"); ::tmpi::check_capture(st, "adam_flat");
  }
  if (advance) adam_advance(step, st);
}

// ============================================================================ fused collectives
// The per-element update is a compile-time policy of the fused kernels: Rule::hyper() reads the step's hyper-parameters once per
// CTA, Rule::update() applies the rule to one float4 of W given the gradient sum, reading and writing the rule's own state (U for
// momentum SGD; M = U region and V for Adam) at element i of the calling rank's arena.
struct SgdRule {
  typedef Hyper Hp;
  static __device__ __forceinline__ Hyper hyper(const FusedArgs& a) { return Hyper{*a.lr_ptr, a.mu, a.inv_k, a.nesterov}; }
  static __device__ __forceinline__ void update(const FusedArgs& a, const Hyper& h, long long i, float4& w, const float4& gsum, int g) {
    float* U = region<float>(a.ctx, a.ctx.rank, a.u_off) + i;
    float4 u = *reinterpret_cast<const float4*>(U);
    sgd4(w, u, gsum, h, a.tab.lr_mult[g], a.tab.wd[g]);
    *reinterpret_cast<float4*>(U) = u;
  }
};
struct AdamRule {
  typedef AdamHyper Hp;
  static __device__ __forceinline__ AdamHyper hyper(const FusedArgs& a) {
    return adam_hyper(a.lr_ptr, a.adam.step, a.inv_k, a.adam.b1, a.adam.b2, a.adam.eps);
  }
  static __device__ __forceinline__ void update(const FusedArgs& a, const AdamHyper& h, long long i, float4& w, const float4& gsum, int g) {
    float* M = region<float>(a.ctx, a.ctx.rank, a.u_off) + i;
    float* V = region<float>(a.ctx, a.ctx.rank, a.adam.v_off) + i;
    float4 m = *reinterpret_cast<const float4*>(M), v = *reinterpret_cast<const float4*>(V);
    adam4(w, m, v, gsum, h, a.tab.lr_mult[g], a.tab.wd[g]);
    *reinterpret_cast<float4*>(M) = m;
    *reinterpret_cast<float4*>(V) = v;
  }
};

// non-exchanged (BN) block: the rank's own gradient, no averaging
template <class Rule>
__device__ __forceinline__ void local_block_update(const FusedArgs& a, const typename Rule::Hp& h, long long b, int g) {
  const long long i = b * kArenaBlock + threadIdx.x * 4;
  float* W = region<float>(a.ctx, a.ctx.rank, a.w_off);
  const float* G = region<float>(a.ctx, a.ctx.rank, a.g_off);
  float4 w = *reinterpret_cast<const float4*>(W + i);
  const float4 gg = *reinterpret_cast<const float4*>(G + i);
  typename Rule::Hp hl = h; hl.inv_k = 1.f;
  Rule::update(a, hl, i, w, gg, g);
  *reinterpret_cast<float4*>(W + i) = w;
  if (a.h_off >= 0) *reinterpret_cast<uint2*>(region<__nv_bfloat16>(a.ctx, a.ctx.rank, a.h_off) + i) = pack_bf16x4(w);
}

// cast the caller's own gradient block to the bf16 wire region
__device__ __forceinline__ void cast_block_to_wire(const FusedArgs& a, long long b) {
  const long long i = b * kArenaBlock + threadIdx.x * 4;
  const float4 gg = *reinterpret_cast<const float4*>(region<float>(a.ctx, a.ctx.rank, a.g_off) + i);
  *reinterpret_cast<uint2*>(region<__nv_bfloat16>(a.ctx, a.ctx.rank, a.wire_off) + i) = pack_bf16x4(gg);
}

__device__ __forceinline__ float4 gather_grad(const FusedArgs& a, long long i) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a.wire16) {
    uint2 v[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) v[p] = ld_sys_u2(region<__nv_bfloat16>(a.ctx, p, a.wire_off) + i);
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) acc = add4(acc, unpack_bf16x4(v[p]));
  } else {
    float4 v[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) v[p] = ld_sys_f4(region<float>(a.ctx, p, a.g_off) + i);
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) acc = add4(acc, v[p]);     // fixed order → bit-identical on all ranks
  }
  return acc;
}

// ---- one-shot: every rank reduces every block itself
// U arena blocks are in flight per CTA iteration (U x world independent 16 B peer loads per thread) — a single
// load per thread cannot cover the ~2 us NVLink round trip.
template <class Rule, int U>
__global__ void __launch_bounds__(kThreads) fused_oneshot_kernel(const FusedArgs a) {
  const typename Rule::Hp h = Rule::hyper(a);
  const long long blo = a.lo / kArenaBlock, bhi = a.hi / kArenaBlock;
  if (a.wire16) {
    for (long long b = blo + blockIdx.x; b < bhi; b += gridDim.x)
      if (a.tab.exch[a.block_group[b]]) cast_block_to_wire(a, b);
  }
  block_barrier(a.ctx);                                  // peers' gradients (or wire copies) are complete
  float* W = region<float>(a.ctx, a.ctx.rank, a.w_off);
  for (long long b0 = blo + blockIdx.x; b0 < bhi; b0 += (long long)gridDim.x * U) {
    float4 gs[U]; int grp[U]; bool ex[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      ex[u] = false; grp[u] = -1;
      if (b < bhi) { grp[u] = a.block_group[b]; ex[u] = a.tab.exch[grp[u]] != 0; }
      if (ex[u]) gs[u] = gather_grad(a, b * kArenaBlock + threadIdx.x * 4);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      if (grp[u] < 0) continue;
      if (!ex[u]) { local_block_update<Rule>(a, h, b, grp[u]); continue; }
      const long long i = b * kArenaBlock + threadIdx.x * 4;
      float4 w = *reinterpret_cast<const float4*>(W + i);
      Rule::update(a, h, i, w, gs[u], grp[u]);
      *reinterpret_cast<float4*>(W + i) = w;
      if (a.h_off >= 0) *reinterpret_cast<uint2*>(region<__nv_bfloat16>(a.ctx, a.ctx.rank, a.h_off) + i) = pack_bf16x4(w);
    }
  }
  block_barrier(a.ctx);                                  // nobody overwrites G while a peer still reads it
}

// ---- two-shot: rank r owns a contiguous slice of the range; reduce → update → push W (+H) to every peer
template <class Rule, int U>
__global__ void __launch_bounds__(kThreads) fused_twoshot_kernel(const FusedArgs a, int use_nvls) {
  const typename Rule::Hp h = Rule::hyper(a);
  const long long blo = a.lo / kArenaBlock, bhi = a.hi / kArenaBlock;
  const long long nb = bhi - blo;
  const long long per = (nb + a.ctx.world - 1) / a.ctx.world;
  const int R = a.ctx.rank, Wn = a.ctx.world;
  if (a.wire16 && !a.pre_reduced) {
    // block b casts, for every owner r, the strip of r's slice that block b of rank r will read
    for (int r = 0; r < Wn; ++r) {
      const long long s0 = blo + r * per, s1 = min(bhi, s0 + per);
      for (long long b = s0 + blockIdx.x; b < s1; b += gridDim.x)
        if (a.tab.exch[a.block_group[b]]) cast_block_to_wire(a, b);
    }
  }
  block_barrier(a.ctx);
  const long long s0 = blo + R * per, s1 = min(bhi, s0 + per);
  float* W = region<float>(a.ctx, R, a.w_off);
  for (long long b0 = s0 + blockIdx.x; b0 < s1; b0 += (long long)gridDim.x * U) {
    float4 gs[U]; int grp[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      grp[u] = -1;
      if (b < s1) { const int g = a.block_group[b]; if (a.tab.exch[g]) grp[u] = g; }
      if (grp[u] >= 0) {
        const long long i = b * kArenaBlock + threadIdx.x * 4;
        if (a.pre_reduced) {
          // the wgrad GEMM epilogues of every rank already red.add-ed their tiles into THIS rank's G (reduce-scatter fused into
          // the producer): consume the sum and clear it for the next step (the closing barrier orders the clear before any
          // peer's next add)
          float* Gl = region<float>(a.ctx, R, a.g_off) + i;
          gs[u] = *reinterpret_cast<const float4*>(Gl);
          *reinterpret_cast<float4*>(Gl) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else if (use_nvls) {
          gs[u] = a.wire16 ? unpack_bf16x4(mc_ld_reduce_bf16x4(reinterpret_cast<char*>(a.ctx.mc_arena) + a.wire_off + i * 2))
                           : mc_ld_reduce_f4(reinterpret_cast<float*>(reinterpret_cast<char*>(a.ctx.mc_arena) + a.g_off) + i);
        } else {
          gs[u] = gather_grad(a, i);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (grp[u] < 0) continue;
      const long long b = b0 + (long long)u * gridDim.x;
      const long long i = b * kArenaBlock + threadIdx.x * 4;
      float4 w = *reinterpret_cast<const float4*>(W + i);
      Rule::update(a, h, i, w, gs[u], grp[u]);
      const uint2 wh = pack_bf16x4(w);
      // owner-keeps-master ships only the bf16 shadow — of plain WEIGHT blocks (group 0).  Biases (and anything else the
      // forward pass reads in fp32 straight from W) always travel as fp32 masters: they are a few KB.
      const bool push_w = a.push_master || a.h_off < 0 || grp[u] != 0;
      if (use_nvls) {
        if (push_w) mc_st_f4(reinterpret_cast<float*>(reinterpret_cast<char*>(a.ctx.mc_arena) + a.w_off) + i, w);
        else *reinterpret_cast<float4*>(W + i) = w;
        if (a.h_off >= 0) mc_st_u2(reinterpret_cast<char*>(a.ctx.mc_arena) + a.h_off + i * 2, wh);
      } else {
#pragma unroll
        for (int p = 0; p < kMaxRanks; ++p) {
          if (p < Wn) {
            if (push_w || p == R) st_f4(region<float>(a.ctx, p, a.w_off) + i, w);
            if (a.h_off >= 0) st_u2(region<__nv_bfloat16>(a.ctx, p, a.h_off) + i, wh);
          }
        }
      }
    }
  }
  // non-exchanged (BN) blocks: every rank updates all of them locally
  for (long long b = blo + blockIdx.x; b < bhi; b += gridDim.x) {
    const int g = a.block_group[b];
    if (!a.tab.exch[g]) local_block_update<Rule>(a, h, b, g);
  }
  block_barrier(a.ctx);                                  // pushed weights are visible everywhere
}

static int pick_grid(long long nblocks, int max_blocks) {
  long long g = std::min<long long>(nblocks, (long long)max_blocks);
  if (g < 1) g = 1;
  if (g > kMaxCommBlocks) g = kMaxCommBlocks;
  return (int)g;
}

// algo: 0 one-shot, 1 two-shot (P2P), 2 two-shot NVLS
template <class Rule>
static void fused_allreduce(const FusedArgs& a, int algo, int max_blocks, cudaStream_t st, const char* name) {
  if (a.lo % kArenaBlock || a.hi % kArenaBlock) throw std::runtime_error(std::string(name) + ": range must be block aligned");
  const long long nb = (a.hi - a.lo) / kArenaBlock;
  if (nb <= 0) return;
  if (algo == 2 && a.ctx.mc_arena == nullptr) throw std::runtime_error(std::string(name) + ": NVLS requested without a multicast mapping");
  const bool wide = a.ctx.world > 4;                     // keep (U x world) peer loads per thread around 8..16
  if (a.pre_reduced && algo == 0) algo = a.ctx.mc_arena ? 2 : 1;     // ownership is the two-shot partition
  if (algo == 0) {
    if (wide) fused_oneshot_kernel<Rule, 2><<<pick_grid(nb, max_blocks), kThreads, 0, st>>>(a);
    else fused_oneshot_kernel<Rule, 4><<<pick_grid(nb, max_blocks), kThreads, 0, st>>>(a);
  } else {
    const long long per = (nb + a.ctx.world - 1) / a.ctx.world;
    const int nv = algo == 2 ? 1 : 0;
    // loads in flight per thread = U (NVLS: one multimem.ld_reduce per block) or U x world (P2P gather).  The exchange runs
    // next to the backward GEMMs on a few dozen co-resident CTAs, so its throughput is (bytes in flight) / (NVLink round trip):
    // keep 8..16 independent 16-byte loads per thread outstanding.  TMPI_FUSED_U overrides (2, 4 or 8).
    static const int u_env = [] { const char* e = getenv("TMPI_FUSED_U"); return e ? atoi(e) : 0; }();
    int U = nv ? 8 : (a.ctx.world <= 2 ? 8 : (wide ? 2 : 4));
    if (u_env == 2 || u_env == 4 || u_env == 8) U = u_env;
    if (U == 8) fused_twoshot_kernel<Rule, 8><<<pick_grid(per, max_blocks), kThreads, 0, st>>>(a, nv);
    else if (U == 4) fused_twoshot_kernel<Rule, 4><<<pick_grid(per, max_blocks), kThreads, 0, st>>>(a, nv);
    else fused_twoshot_kernel<Rule, 2><<<pick_grid(per, max_blocks), kThreads, 0, st>>>(a, nv);
  }
  count_launch(); TMPI_CHECK_LAUNCH(name); ::tmpi::check_capture(st, name);
}

void fused_allreduce_sgd(const FusedArgs& a, int algo, int max_blocks, cudaStream_t st) {
  fused_allreduce<SgdRule>(a, algo, max_blocks, st, "fused_allreduce_sgd");
}

void fused_allreduce_adam(const FusedArgs& a, int algo, int max_blocks, cudaStream_t st) {
  if (a.pre_reduced) throw std::runtime_error("fused_allreduce_adam: gradients reduce-scattered by the GEMM epilogue are not supported");
  if (a.adam.step == nullptr) throw std::runtime_error("fused_allreduce_adam: no step counter");
  fused_allreduce<AdamRule>(a, algo, max_blocks, st, "fused_allreduce_adam");
}

// every rank pushes the slice it owns (two-shot partition of [lo, hi)) of the fp32 region at byte offset `off` to all peers:
// re-synchronises W after steps that ran with push_master = 0, and the optimizer state (momentum / Adam moments) that two-shot
// steps update on the owner only (before a checkpoint / weight averaging / anything that reads them on a non-owner)
__global__ void __launch_bounds__(kThreads) push_region_kernel(const FusedArgs a, long long off) {
  const long long blo = a.lo / kArenaBlock, bhi = a.hi / kArenaBlock;
  const long long per = (bhi - blo + a.ctx.world - 1) / a.ctx.world;
  const int R = a.ctx.rank;
  const long long s0 = blo + R * per, s1 = min(bhi, s0 + per);
  block_barrier(a.ctx);
  const float* X = region<float>(a.ctx, R, off);
  for (long long b = s0 + blockIdx.x; b < s1; b += gridDim.x) {
    if (!a.tab.exch[a.block_group[b]]) continue;
    const long long i = b * kArenaBlock + threadIdx.x * 4;
    const float4 x = *reinterpret_cast<const float4*>(X + i);
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p)
      if (p < a.ctx.world && p != R) st_f4(region<float>(a.ctx, p, off) + i, x);
  }
  block_barrier(a.ctx);
}
void push_region_slices(const FusedArgs& a, long long off, int max_blocks, cudaStream_t st) {
  if (a.lo % kArenaBlock || a.hi % kArenaBlock) throw std::runtime_error("push_region_slices: range must be block aligned");
  const long long nb = (a.hi - a.lo) / kArenaBlock;
  if (nb <= 0) return;
  const long long per = (nb + a.ctx.world - 1) / a.ctx.world;
  push_region_kernel<<<pick_grid(per, max_blocks), kThreads, 0, st>>>(a, off);
  count_launch(); TMPI_CHECK_LAUNCH("push_region_slices"); ::tmpi::check_capture(st, "push_region_slices");
}

// ============================================================================ plain flat allreduce (sum * scale) src region → dst region
__global__ void __launch_bounds__(kThreads) allreduce_oneshot_kernel(const ReduceArgs a) {
  const long long blo = a.lo / kArenaBlock, bhi = a.hi / kArenaBlock;
  block_barrier(a.ctx);
  float* D = region<float>(a.ctx, a.ctx.rank, a.dst_off);
  for (long long b = blo + blockIdx.x; b < bhi; b += gridDim.x) {
    if (a.skip_local_groups && !a.tab.exch[a.block_group[b]]) continue;
    const long long i = b * kArenaBlock + threadIdx.x * 4;
    float4 v[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) v[p] = ld_sys_f4(region<float>(a.ctx, p, a.src_off) + i);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) acc = add4(acc, v[p]);
    acc.x *= a.scale; acc.y *= a.scale; acc.z *= a.scale; acc.w *= a.scale;
    *reinterpret_cast<float4*>(D + i) = acc;
    if (a.h_off >= 0) *reinterpret_cast<uint2*>(region<__nv_bfloat16>(a.ctx, a.ctx.rank, a.h_off) + i) = pack_bf16x4(acc);
  }
  block_barrier(a.ctx);
}

__global__ void __launch_bounds__(kThreads) allreduce_twoshot_kernel(const ReduceArgs a, int use_nvls) {
  const long long blo = a.lo / kArenaBlock, bhi = a.hi / kArenaBlock;
  const long long per = (bhi - blo + a.ctx.world - 1) / a.ctx.world;
  const long long s0 = blo + a.ctx.rank * per, s1 = min(bhi, s0 + per);
  block_barrier(a.ctx);
  for (long long b = s0 + blockIdx.x; b < s1; b += gridDim.x) {
    if (a.skip_local_groups && !a.tab.exch[a.block_group[b]]) continue;
    const long long i = b * kArenaBlock + threadIdx.x * 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (use_nvls) {
      acc = mc_ld_reduce_f4(reinterpret_cast<float*>(reinterpret_cast<char*>(a.ctx.mc_arena) + a.src_off) + i);
    } else {
      float4 v[kMaxRanks];
#pragma unroll
      for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) v[p] = ld_sys_f4(region<float>(a.ctx, p, a.src_off) + i);
#pragma unroll
      for (int p = 0; p < kMaxRanks; ++p) if (p < a.ctx.world) acc = add4(acc, v[p]);
    }
    acc.x *= a.scale; acc.y *= a.scale; acc.z *= a.scale; acc.w *= a.scale;
    const uint2 hh = pack_bf16x4(acc);
    if (use_nvls) {
      mc_st_f4(reinterpret_cast<float*>(reinterpret_cast<char*>(a.ctx.mc_arena) + a.dst_off) + i, acc);
      if (a.h_off >= 0) mc_st_u2(reinterpret_cast<char*>(a.ctx.mc_arena) + a.h_off + i * 2, hh);
    } else {
#pragma unroll
      for (int p = 0; p < kMaxRanks; ++p) {
        if (p < a.ctx.world) {
          st_f4(region<float>(a.ctx, p, a.dst_off) + i, acc);
          if (a.h_off >= 0) st_u2(region<__nv_bfloat16>(a.ctx, p, a.h_off) + i, hh);
        }
      }
    }
  }
  block_barrier(a.ctx);
}

void allreduce_flat(const ReduceArgs& a, int algo, int max_blocks, cudaStream_t st) {
  if (a.lo % kArenaBlock || a.hi % kArenaBlock) throw std::runtime_error("allreduce_flat: range must be block aligned");
  const long long nb = (a.hi - a.lo) / kArenaBlock;
  if (nb <= 0) return;
  if (algo == 0 && a.src_off == a.dst_off) throw std::runtime_error("allreduce_flat: one-shot cannot run in place");
  if (algo == 2 && a.ctx.mc_arena == nullptr) throw std::runtime_error("allreduce_flat: NVLS requested without a multicast mapping");
  if (algo == 0) allreduce_oneshot_kernel<<<pick_grid(nb, max_blocks), kThreads, 0, st>>>(a);
  else allreduce_twoshot_kernel<<<pick_grid((nb + a.ctx.world - 1) / a.ctx.world, max_blocks), kThreads, 0, st>>>(a, algo == 2 ? 1 : 0);
  count_launch(); TMPI_CHECK_LAUNCH("allreduce_flat"); ::tmpi::check_capture(st, "allreduce_flat");
}

// standalone device barrier (tests / stream alignment)
__global__ void barrier_kernel(const CommCtx c) { block_barrier(c); }
void device_barrier(const CommCtx& c, cudaStream_t st) {
  barrier_kernel<<<1, 32, 0, st>>>(c);
  count_launch(); TMPI_CHECK_LAUNCH("device_barrier"); ::tmpi::check_capture(st, "device_barrier");
}

// ============================================================================ device-side protocol words
// The 4 KiB tail of every rank's signal pad (peer-mapped like the rest of it) holds the words of the asynchronous rules:
//   [0] EASGD next ticket   [1] EASGD now serving   [2] EASGD exchanges served
//   [32 + 2*src], [33 + 2*src]   GOSGD inbox slot of sender `src`: {sequence number, push-sum weight bits}
//   [96 + dst]                   GOSGD acknowledgements: receiver `dst` writes the sequence number it merged (on the SENDER's pad)
__device__ __forceinline__ uint32_t* proto_words(const CommCtx& c, int p) {
  return c.sig[p] + (size_t)kMaxCommBlocks * kMaxRanks + kMaxCommBlocks;
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
  uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_release_sys_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_add_sys_v4(float* p, float4 v) {
  asm volatile("red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ============================================================================ EASGD elastic exchange (worker side, center over NVLink)
// Reference: the server serialises workers with a blocking MPI recv and both sides broadcast their full model
// (easgd_server.py:152-164, lib/exchanger.py:214-261).  Here the workers queue on the DEVICE: a ticket lock in the center
// rank's signal pad (atom.acq_rel.sys take, st.release.sys hand-over) brackets ONE kernel on the worker's GPU that reads the
// center over NVLink, computes d = α(w − c) and updates both sides.  Three stream-ordered launches (acquire → elastic →
// release) instead of a grid-wide sync inside one kernel: no co-residency requirement, graph-capturable, and the host never
// waits.  lockfree = 1: no lock at all — the center update is a vector red.add (commutative, so no update can be lost) and
// the workers run fully concurrently.
__global__ void ticket_acquire_kernel(CommCtx c, int owner, uint32_t* local) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  uint32_t* lock = proto_words(c, owner);
  uint32_t my;
  asm volatile("atom.acq_rel.sys.global.add.u32 %0, [%1], 1;" : "=r"(my) : "l"(lock) : "memory");
  local[0] = my;
  const long long t0 = clock64();
  while (ld_acquire_sys_u32(lock + 1) != my) {
    if (clock64() - t0 > c.spin_limit) __trap();
    __nanosleep(200);
  }
}
__global__ void ticket_release_kernel(CommCtx c, int owner, uint32_t* local) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  uint32_t* lock = proto_words(c, owner);
  __threadfence_system();
  asm volatile("red.relaxed.sys.global.add.u32 [%0], 1;" ::"l"(lock + 2) : "memory");
  st_release_sys_u32(lock + 1, local[0] + 1u);
}

// U arena blocks in flight per CTA iteration: U independent 16 B NVLink loads per thread cover the ~2 us round trip
template <int U>
__global__ void __launch_bounds__(kThreads) easgd_elastic_kernel(float* __restrict__ w, __nv_bfloat16* __restrict__ h, float* c /*peer*/,
                                                                 float alpha, long long nblk, int lockfree) {
  for (long long b0 = blockIdx.x; b0 < nblk; b0 += (long long)gridDim.x * U) {
    float4 cv[U], wv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      if (b < nblk) {
        const long long i = b * kArenaBlock + threadIdx.x * 4;
        cv[u] = ld_sys_f4(c + i);
        wv[u] = *reinterpret_cast<const float4*>(w + i);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      if (b >= nblk) continue;
      const long long i = b * kArenaBlock + threadIdx.x * 4;
      const float4 d = make_float4(alpha * (wv[u].x - cv[u].x), alpha * (wv[u].y - cv[u].y), alpha * (wv[u].z - cv[u].z),
                                   alpha * (wv[u].w - cv[u].w));
      wv[u].x -= d.x; wv[u].y -= d.y; wv[u].z -= d.z; wv[u].w -= d.w;
      *reinterpret_cast<float4*>(w + i) = wv[u];
      if (h) *reinterpret_cast<uint2*>(h + i) = pack_bf16x4(wv[u]);
      if (lockfree) red_add_sys_v4(c + i, d);
      else st_f4(c + i, add4(cv[u], d));
    }
  }
  __threadfence_system();
}

void easgd_elastic(void* w, void* h, void* center, float alpha, long long n, int max_blocks, int lockfree, cudaStream_t st) {
  if (n % kArenaBlock) throw std::runtime_error("easgd_elastic: n must be block aligned");
  const long long nb = n / kArenaBlock;
  if (nb <= 0) return;
  easgd_elastic_kernel<4><<<pick_grid((nb + 3) / 4, max_blocks), kThreads, 0, st>>>((float*)w, (__nv_bfloat16*)h, (float*)center, alpha, nb,
                                                                                lockfree);
  count_launch(); TMPI_CHECK_LAUNCH("easgd_elastic"); ::tmpi::check_capture(st, "easgd_elastic");
}
void ticket_acquire(const CommCtx& c, int owner, void* local_state, cudaStream_t st) {
  ticket_acquire_kernel<<<1, 32, 0, st>>>(c, owner, (uint32_t*)local_state);
  count_launch(); TMPI_CHECK_LAUNCH("ticket_acquire"); ::tmpi::check_capture(st, "ticket_acquire");
}
void ticket_release(const CommCtx& c, int owner, void* local_state, cudaStream_t st) {
  ticket_release_kernel<<<1, 32, 0, st>>>(c, owner, (uint32_t*)local_state);
  count_launch(); TMPI_CHECK_LAUNCH("ticket_release"); ::tmpi::check_capture(st, "ticket_release");
}

// dst = src (+ bf16 shadow) over peer memory: EASGD copy_to_local, GOSGD snapshot.  `gate` (optional, device word): the copy
// runs only when *gate != 0 (GOSGD: the push was admitted by gosgd_push_begin).
template <int U>
__global__ void __launch_bounds__(kThreads) copy_flat_kernel(float* dst, __nv_bfloat16* dst_h, const float* src, long long nblk,
                                                             const uint32_t* __restrict__ gate) {
  if (gate && *gate == 0u) return;
  for (long long b0 = blockIdx.x; b0 < nblk; b0 += (long long)gridDim.x * U) {
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      if (b < nblk) v[u] = ld_sys_f4(src + b * kArenaBlock + threadIdx.x * 4);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long b = b0 + (long long)u * gridDim.x;
      if (b >= nblk) continue;
      const long long i = b * kArenaBlock + threadIdx.x * 4;
      st_f4(dst + i, v[u]);
      if (dst_h) *reinterpret_cast<uint2*>(dst_h + i) = pack_bf16x4(v[u]);
    }
  }
  __threadfence_system();
}
void copy_flat(void* dst, void* dst_h, const void* src, long long n, int max_blocks, const void* gate, cudaStream_t st) {
  if (n % kArenaBlock) throw std::runtime_error("copy_flat: n must be block aligned");
  const long long nb = n / kArenaBlock;
  if (nb <= 0) return;
  copy_flat_kernel<4><<<pick_grid((nb + 3) / 4, max_blocks), kThreads, 0, st>>>((float*)dst, (__nv_bfloat16*)dst_h, (const float*)src, nb,
                                                                            (const uint32_t*)gate);
  count_launch(); TMPI_CHECK_LAUNCH("copy_flat"); ::tmpi::check_capture(st, "copy_flat");
}

// ============================================================================ GOSGD:  w ← (a_self·w + a_src·b) / (a_self + a_src)
// Host-driven form (CPU-mirrored semantics, tests): coefficients passed by value, `b` = local mailbox or a peer's snapshot.
template <int U>
__global__ void __launch_bounds__(kThreads) gosgd_merge_kernel(float* __restrict__ w, __nv_bfloat16* __restrict__ h, const float* b,
                                                               float ca, float cb, long long nblk) {
  for (long long b0 = blockIdx.x; b0 < nblk; b0 += (long long)gridDim.x * U) {
    float4 bv[U], wv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long blk = b0 + (long long)u * gridDim.x;
      if (blk < nblk) {
        const long long i = blk * kArenaBlock + threadIdx.x * 4;
        bv[u] = ld_sys_f4(b + i);
        wv[u] = *reinterpret_cast<const float4*>(w + i);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long blk = b0 + (long long)u * gridDim.x;
      if (blk >= nblk) continue;
      const long long i = blk * kArenaBlock + threadIdx.x * 4;
      float4 o;
      o.x = ca * wv[u].x + cb * bv[u].x; o.y = ca * wv[u].y + cb * bv[u].y; o.z = ca * wv[u].z + cb * bv[u].z; o.w = ca * wv[u].w + cb * bv[u].w;
      *reinterpret_cast<float4*>(w + i) = o;
      if (h) *reinterpret_cast<uint2*>(h + i) = pack_bf16x4(o);
    }
  }
}
void gosgd_merge(void* w, void* h, const void* b, float a_self, float a_src, long long n, int max_blocks, cudaStream_t st) {
  if (n % kArenaBlock) throw std::runtime_error("gosgd_merge: n must be block aligned");
  const long long nb = n / kArenaBlock;
  if (nb <= 0) return;
  const float inv = 1.f / (a_self + a_src);
  gosgd_merge_kernel<4><<<pick_grid((nb + 3) / 4, max_blocks), kThreads, 0, st>>>((float*)w, (__nv_bfloat16*)h, (const float*)b, a_self * inv,
                                                                              a_src * inv, nb);
  count_launch(); TMPI_CHECK_LAUNCH("gosgd_merge"); ::tmpi::check_capture(st, "gosgd_merge");
}

// ---- device-side gossip protocol (no host message, no stream synchronisation on the path; ref lib/exchanger.py:484-584
//      blocks the sender inside ncclBcast until the receiver joins).
// Local state words (uint32 / float bits, one small device buffer per rank):
//   [0] alpha (float)  [1] push admitted flag  [2] last dest (+1; 0 = none)  [3] sequence of the outstanding push
//   [4] pushes done    [5] pushes skipped (previous snapshot still being pulled)  [6] merges done
//   [8] merge: chosen src (+1; 0 = none)  [9] merge: src's sequence  [10] ca (float)  [11] cb (float)
//   [16 + src] last sequence merged from src        [32 + dst] sequence counter of pushes sent to dst
__global__ void gosgd_push_begin_kernel(CommCtx c, uint32_t* st) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  uint32_t ok = 1u;
  const uint32_t last = st[2];
  if (last != 0u) {
    // my snapshot region is single-buffered: the previous receiver must have pulled it (it acknowledges on MY pad)
    const uint32_t acked = ld_acquire_sys_u32(proto_words(c, c.rank) + 96 + (last - 1u));
    if (acked != st[3]) ok = 0u;
  }
  st[1] = ok;
  if (ok) {
    float a = __uint_as_float(st[0]) * 0.5f;                    // push-sum: keep half, ship half
    st[0] = __float_as_uint(a);
  } else {
    st[5] += 1u;
  }
}
__global__ void gosgd_push_end_kernel(CommCtx c, uint32_t* st, int dest) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (st[1] == 0u) return;
  __threadfence_system();                                       // the snapshot (copy_flat before me on this stream) is visible
  const uint32_t seq = st[32 + dest] + 1u;
  st[32 + dest] = seq; st[2] = (uint32_t)dest + 1u; st[3] = seq; st[4] += 1u;
  uint32_t* inbox = proto_words(c, dest) + 32 + 2 * c.rank;
  asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(inbox + 1), "r"(st[0]) : "memory");     // shipped weight = what I kept
  st_release_sys_u32(inbox, seq);
}
// receiver: pick at most one pending push (lowest rank first, fair enough for p << 1)
__global__ void gosgd_poll_kernel(CommCtx c, uint32_t* st) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  st[8] = 0u;
  const uint32_t* inbox = proto_words(c, c.rank) + 32;
  for (int s = 0; s < c.world; ++s) {
    if (s == c.rank) continue;
    const uint32_t seq = ld_acquire_sys_u32(inbox + 2 * s);
    if (seq != st[16 + s]) {
      const float a_src = __uint_as_float(ld_acquire_sys_u32(inbox + 2 * s + 1));
      const float a_self = __uint_as_float(st[0]);
      const float inv = 1.f / (a_self + a_src);
      st[8] = (uint32_t)s + 1u; st[9] = seq;
      st[10] = __float_as_uint(a_self * inv); st[11] = __float_as_uint(a_src * inv);
      st[0] = __float_as_uint(a_self + a_src);
      return;
    }
  }
}
template <int U>
__global__ void __launch_bounds__(kThreads) gosgd_pull_merge_kernel(CommCtx c, const uint32_t* __restrict__ st, long long w_off, long long h_off,
                                                                    long long snap_off, long long nblk) {
  const uint32_t chosen = st[8];
  if (chosen == 0u) return;
  const int src = (int)chosen - 1;
  const float ca = __uint_as_float(st[10]), cb = __uint_as_float(st[11]);
  float* w = region<float>(c, c.rank, w_off);
  __nv_bfloat16* h = h_off >= 0 ? region<__nv_bfloat16>(c, c.rank, h_off) : nullptr;
  const float* b = region<float>(c, src, snap_off);
  for (long long b0 = blockIdx.x; b0 < nblk; b0 += (long long)gridDim.x * U) {
    float4 bv[U], wv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long blk = b0 + (long long)u * gridDim.x;
      if (blk < nblk) {
        const long long i = blk * kArenaBlock + threadIdx.x * 4;
        bv[u] = ld_sys_f4(b + i);
        wv[u] = *reinterpret_cast<const float4*>(w + i);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long blk = b0 + (long long)u * gridDim.x;
      if (blk >= nblk) continue;
      const long long i = blk * kArenaBlock + threadIdx.x * 4;
      float4 o;
      o.x = ca * wv[u].x + cb * bv[u].x; o.y = ca * wv[u].y + cb * bv[u].y; o.z = ca * wv[u].z + cb * bv[u].z; o.w = ca * wv[u].w + cb * bv[u].w;
      *reinterpret_cast<float4*>(w + i) = o;
      if (h) *reinterpret_cast<uint2*>(h + i) = pack_bf16x4(o);
    }
  }
}
__global__ void gosgd_ack_kernel(CommCtx c, uint32_t* st) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const uint32_t chosen = st[8];
  if (chosen == 0u) return;
  const int src = (int)chosen - 1;
  st[16 + src] = st[9]; st[6] += 1u; st[8] = 0u;
  __threadfence_system();
  st_release_sys_u32(proto_words(c, src) + 96 + c.rank, st[9]);       // the sender may overwrite its snapshot now
}

void gosgd_push(const CommCtx& c, void* state, int dest, long long w_off, long long snap_off, long long n, int max_blocks, cudaStream_t st) {
  if (n % kArenaBlock) throw std::runtime_error("gosgd_push: n must be block aligned");
  if (dest < 0 || dest >= c.world || dest == c.rank) throw std::runtime_error("gosgd_push: bad destination");
  uint32_t* s = (uint32_t*)state;
  gosgd_push_begin_kernel<<<1, 32, 0, st>>>(c, s);
  char* base = reinterpret_cast<char*>(c.arena[c.rank]);
  const long long nb = n / kArenaBlock;
  copy_flat_kernel<4><<<pick_grid((nb + 3) / 4, max_blocks), kThreads, 0, st>>>((float*)(base + snap_off), nullptr, (const float*)(base + w_off), nb,
                                                                            s + 1);
  gosgd_push_end_kernel<<<1, 32, 0, st>>>(c, s, dest);
  count_launch(3); TMPI_CHECK_LAUNCH("gosgd_push"); ::tmpi::check_capture(st, "gosgd_push");
}
void gosgd_poll_merge(const CommCtx& c, void* state, long long w_off, long long h_off, long long snap_off, long long n, int max_blocks,
                      cudaStream_t st) {
  if (n % kArenaBlock) throw std::runtime_error("gosgd_poll_merge: n must be block aligned");
  uint32_t* s = (uint32_t*)state;
  const long long nb = n / kArenaBlock;
  gosgd_poll_kernel<<<1, 32, 0, st>>>(c, s);
  gosgd_pull_merge_kernel<4><<<pick_grid((nb + 3) / 4, max_blocks), kThreads, 0, st>>>(c, s, w_off, h_off, snap_off, nb);
  gosgd_ack_kernel<<<1, 32, 0, st>>>(c, s);
  count_launch(3); TMPI_CHECK_LAUNCH("gosgd_poll_merge"); ::tmpi::check_capture(st, "gosgd_poll_merge");
}

// ============================================================================ reference kernels K1..K5 (legacy strategies)
template <typename TI, typename TO> __global__ void cast_kernel(const TI* __restrict__ s, TO* __restrict__ d, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) d[i] = (TO)(float)s[i];
}
// kind: 0 f32→f16, 1 f16→f32, 2 f32→bf16, 3 bf16→f32     (K1/K5: float2half / half2float)
void cast_flat(const void* src, void* dst, long long n, int kind, cudaStream_t st) {
  const int g = (int)std::min<long long>((n + 255) / 256, (long long)sm_count() * 16);
  if (n <= 0) return;
  switch (kind) {
    case 0: cast_kernel<float, __half><<<g, 256, 0, st>>>((const float*)src, (__half*)dst, n); break;
    case 1: cast_kernel<__half, float><<<g, 256, 0, st>>>((const __half*)src, (float*)dst, n); break;
    case 2: cast_kernel<float, __nv_bfloat16><<<g, 256, 0, st>>>((const float*)src, (__nv_bfloat16*)dst, n); break;
    case 3: cast_kernel<__nv_bfloat16, float><<<g, 256, 0, st>>>((const __nv_bfloat16*)src, (float*)dst, n); break;
    default: throw std::runtime_error("cast_flat: bad kind");
  }
  count_launch(); TMPI_CHECK_LAUNCH("cast_flat"); ::tmpi::check_capture(st, "cast_flat");
}

// K2/K3 sumfloats / sumhalfs with the reference's loop bug fixed (SURVEY §2.9 #1): dst[i] = Σ_j src[i + chunk*j], fp32 accumulate
template <typename T> __global__ void sum_chunks_kernel(const T* __restrict__ s, T* __restrict__ d, long long chunk, int nchunks) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < chunk; i += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j < nchunks; ++j) acc += (float)s[i + chunk * j];
    d[i] = (T)acc;
  }
}
void sum_chunks(const void* src, void* dst, long long chunk, int nchunks, int is_half, cudaStream_t st) {
  if (chunk <= 0) return;
  const int g = (int)std::min<long long>((chunk + 255) / 256, (long long)sm_count() * 16);
  if (is_half) sum_chunks_kernel<__half><<<g, 256, 0, st>>>((const __half*)src, (__half*)dst, chunk, nchunks);
  else sum_chunks_kernel<float><<<g, 256, 0, st>>>((const float*)src, (float*)dst, chunk, nchunks);
  count_launch(); TMPI_CHECK_LAUNCH("sum_chunks"); ::tmpi::check_capture(st, "sum_chunks");
}

// K4/K5 vecadd / vecaddhalf: cur[i] += tmp[i]
template <typename T> __global__ void vecadd_kernel(T* __restrict__ cur, const T* __restrict__ tmp, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    cur[i] = (T)((float)cur[i] + (float)tmp[i]);
}
void vecadd(void* cur, const void* tmp, long long n, int is_half, cudaStream_t st) {
  if (n <= 0) return;
  const int g = (int)std::min<long long>((n + 255) / 256, (long long)sm_count() * 16);
  if (is_half) vecadd_kernel<__half><<<g, 256, 0, st>>>((__half*)cur, (const __half*)tmp, n);
  else vecadd_kernel<float><<<g, 256, 0, st>>>((float*)cur, (const float*)tmp, n);
  count_launch(); TMPI_CHECK_LAUNCH("vecadd"); ::tmpi::check_capture(st, "vecadd");
}

}  // namespace tmpi
