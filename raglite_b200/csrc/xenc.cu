// BERT cross-encoder forward (ms-marco-MiniLM-L-12 and BERT-base geometries) for sm_100a: the arithmetic behind
// rerank_chunks (reference _search.py:364-397 -> rerankers FlashRankRanker -> onnxruntime, all
// third-party).  Variable-length packed batches (no padding): tokens [T, H], cu_seqlens [P + 1].
//
//   embed_ln_kernel      word + position + token-type embeddings, LayerNorm          (fp32 math, fp16 out)
//   linear_tcgen05_kernel  Y = act(X W^T + b): tcgen05.mma (M=128 tokens, N<=256 outputs per pass, K
//                        sliced by 64), X copied into 128B-swizzled smem by loader warps, W as a
//                        pre-swizzled fp16 image fetched with cp.async.bulk, fp32 accumulate in TMEM,
//                        bias / GELU(erf) fused in the TMEM epilogue
//   attention2_kernel    softmax(Q K^T / sqrt(dh)) V per (sequence, head), fp32 math, head_dim 32
//   attention64_kernel   the same for head_dim 64 (BERT-base), K / V streamed through a cp.async ring
//   add_ln_kernel        LayerNorm(x + residual)
//   cls_head_kernel      pooler (dense + tanh on [CLS]) -> classifier -> logit, sigmoid score
#include <cuda.h>
#include <cuda_fp16.h>

#include <type_traits>

#include <mutex>

#include "common.cuh"
#include "tcgen05_ptx.cuh"

namespace rl {
namespace {

using namespace tc;

constexpr int kTileM = 128;
constexpr int kSliceK = 64;
constexpr int kMaxN = 256;
constexpr int kNumEpiWarps = 8;   // warp w reads TMEM lane quarter w % 4; warps 4..7 take the odd 32-column chunks
constexpr int kMmaWarp = 8;
constexpr int kWWarp = 9;
constexpr int kFirstLoaderWarp = 10;
constexpr int kNumLoaderWarps = 8;
constexpr int kLoadDepth = 3;     // activation K-slices in flight per loader thread (registers)
constexpr uint32_t kBarBytes = 256;                         // mbarriers + TMEM base pointer
constexpr uint32_t kEpiPitch = 80;                          // bytes per staged row: 64 B of fp16 + pad (conflict-free 16 B stores)
constexpr uint32_t kEpiWarpBytes = 32 * kEpiPitch;          // one 32 x 32 output chunk per epilogue warp
constexpr uint32_t kEpiBytes = kNumEpiWarps * kEpiWarpBytes;
constexpr int kThreads = (kFirstLoaderWarp + kNumLoaderWarps) * 32;
constexpr int kMaxStages = 8;
constexpr int kABytes = kTileM * 128;
constexpr uint32_t kSmemBudget = 226 * 1024;

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// GELU(x) = x/2 (1 + erf(x / sqrt 2)) with erfc from Abramowitz & Stegun 7.1.28,
// 1 - erf(z) = (1 + a1 z + ... + a6 z^6)^-16 (|error| <= 3e-7; 8e-7 on the GELU value in float32, far
// below the fp16 rounding of the stored activation): 6 FMAs, 4 squarings and ONE special-function op.
// The epilogue is bound by the ALU / MUFU pipes, so the instruction count per element is what counts.
__device__ __forceinline__ float gelu_erf(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float p = fmaf(0.0000430638f, z, 0.0002765672f);
  p = fmaf(p, z, 0.0001520143f);
  p = fmaf(p, z, 0.0092705272f);
  p = fmaf(p, z, 0.0422820123f);
  p = fmaf(p, z, 0.0705230784f);
  p = fmaf(p, z, 1.f);
  p *= p; p *= p; p *= p; p *= p;   // p^16 (overflows to +inf for huge z: the tail is then exactly 0)
  float tail;                       // 1 - erf(z), z >= 0
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(tail) : "f"(p));
  const float half_x = 0.5f * x;
  // x >= 0: x/2 (2 - tail);  x < 0: x/2 tail
  return half_x * (x >= 0.f ? 2.f - tail : tail);
}

// ---- weight image: W[N, K] fp32 row-major -> per (pass, k-slice) swizzled fp16 UMMA B tiles -------------
// Output columns per pass.  Short-K layers whose width is a multiple of 192 (QKV, out-proj, FFN-up of the
// MiniLM shapes: K = 384, N = 1152 / 384 / 1536) use 192-column passes: the whole K extent of such a pass
// (192 x 384 fp16 = 144 KB) stays RESIDENT in shared memory while the CTA walks the token tiles
// (linear_wres_kernel).  Everything else streams 256-column weight slices (linear_tcgen05_kernel).
constexpr int kResN = 192;
constexpr int kResMaxKs = 6;
__host__ __device__ inline bool use_resident(int N, int K) { return K % kSliceK == 0 && K / kSliceK <= kResMaxKs && N % kResN == 0; }
__host__ __device__ inline int pass_width(int N, int K) { return use_resident(N, K) ? kResN : kMaxN; }

__host__ __device__ inline int pass_rows(int N, int pass, int pw = kMaxN) {
  const int rem = N - pass * pw;
  return rem < pw ? rem : pw;
}
__host__ __device__ inline size_t pass_offset_halves(int N, int K, int pass, int pw = kMaxN) {
  const int n_ks = (K + kSliceK - 1) / kSliceK;
  return (size_t)pass * pw * n_ks * kSliceK;  // full passes precede; only the last pass is short
}

__global__ void pack_linear_kernel(const float* __restrict__ W, int N, int K, int pw, __half* __restrict__ img) {
  const int n_ks = (K + kSliceK - 1) / kSliceK;
  const int64_t total = (int64_t)((N + 15) / 16 * 16) * n_ks * kSliceK;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(idx / (n_ks * kSliceK));
    const int kk = (int)(idx % (n_ks * kSliceK));
    const int pass = n / pw, r = n % pw;
    const int nb = (pass_rows(N, pass, pw) + 15) / 16 * 16;
    const int ks = kk / kSliceK, e = kk % kSliceK;
    const float v = (n < N && kk < K) ? W[(size_t)n * K + kk] : 0.f;
    const size_t off = pass_offset_halves(N, K, pass, pw) + ((size_t)ks * nb + r) * kSliceK +
                       (size_t)((((e >> 3) ^ (r & 7)) << 3) + (e & 7));
    img[off] = __float2half_rn(v);
  }
}

// ---- tcgen05 linear layer ---------------------------------------------------------------------------------
struct LinArgs {
  const __half* X;     // [T, K]
  const __half* img;   // packed weights
  const float* bias;   // [N]
  __half* Y;           // [T, N]
  int T, N, K, act;    // act: 0 none, 1 GELU(erf)
  int n_pass, n_ks, stages;
  int cp_async;        // 1: activation tile through cp.async (launch_linear); 0: the register ring
  int pw;              // output columns per pass of the weight image (pass_width(N, K))
};

// 16-byte asynchronous global -> shared copy (zero-fills when src_bytes == 0) and the mbarrier arrive
// that fires once all of this thread's earlier cp.async have landed.
__device__ __forceinline__ void cp_async_16(uint32_t dst_smem, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__host__ __device__ inline uint32_t lin_stage_bytes() { return kABytes + kMaxN * 128u; }

__global__ void __launch_bounds__(kThreads, 1) linear_tcgen05_kernel(const LinArgs t) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const uint32_t sbytes = lin_stage_bytes();
  uint64_t* full = reinterpret_cast<uint64_t*>(base + (size_t)t.stages * sbytes);
  uint64_t* empty = full + kMaxStages;
  uint64_t* tmem_full = empty + kMaxStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  unsigned char* epi_stage = base + (size_t)t.stages * sbytes + kBarBytes;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (t.T + kTileM - 1) / kTileM;
  // item = m_tile * n_pass + pass
  const int64_t n_items = (int64_t)m_tiles * t.n_pass;
  const int64_t first = blockIdx.x, stride = gridDim.x;
  const int64_t my_items = first < n_items ? (n_items - first + stride - 1) / stride : 0;
  auto tile_of = [&](int64_t item) -> int { return (int)(item / t.n_pass); };

  if (threadIdx.x == 0) {
    for (int i = 0; i < t.stages; ++i) {
      mbar_init(&full[i], (t.cp_async ? kNumLoaderWarps * 32 : kNumLoaderWarps) + 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], kNumEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp >= kFirstLoaderWarp) {
    // activations: fp16 rows -> swizzled K-major smem tile (UMMA A), 4 x 16-byte chunks per thread and
    // slice.  The loads of kLoadDepth slices are in flight at once (a register ring that runs across
    // item boundaries): one memory latency per slice would otherwise bound the whole kernel.
    const int lt = threadIdx.x - kFirstLoaderWarp * 32;
    const int j = lt & 7, r0 = lt >> 3;  // chunk j of rows r0 + 32 i
    const int64_t n_slices = my_items * t.n_ks;
    auto issue = [&](int64_t g, uint4 (&v)[4]) {
      if (g >= n_slices) return;
      const int64_t it = g / t.n_ks;
      const int ks = (int)(g - it * t.n_ks);
      const int m_tile = tile_of(first + it * stride);
      const int col = ks * kSliceK + j * 8;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = m_tile * kTileM + r0 + 32 * i;
        v[i] = make_uint4(0u, 0u, 0u, 0u);
        if (row < t.T && col < t.K) v[i] = __ldg(reinterpret_cast<const uint4*>(t.X + (size_t)row * t.K + col));
      }
    };
    int stage = 0;
    uint32_t phase = 0;
    auto commit = [&](int64_t g, const uint4 (&v)[4]) {
      if (g >= n_slices) return;
      mbar_wait(&empty[stage], phase ^ 1u);
      unsigned char* A = base + (size_t)stage * sbytes;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = r0 + 32 * i;
        *reinterpret_cast<uint4*>(A + (uint32_t)r * 128u + (((uint32_t)j ^ ((uint32_t)r & 7u)) << 4)) = v[i];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[stage]);
      if (++stage == t.stages) { stage = 0; phase ^= 1u; }
    };
    if (t.cp_async) {
      // Each thread fires its four 16-byte copies straight into the swizzled tile and lets the hardware arrive on
      // the stage's barrier when they land, so the loaders run ahead by as many stages as are free instead of by
      // the depth of a register ring (352 vs 309 us for a layer's four GEMMs, profiles/r01_linear_loader_ab.json).
      for (int64_t g = 0; g < n_slices; ++g) {
        const int64_t it = g / t.n_ks;
        const int ks = (int)(g - it * t.n_ks);
        const int m_tile = tile_of(first + it * stride);
        const int col = ks * kSliceK + j * 8;
        mbar_wait(&empty[stage], phase ^ 1u);
        const uint32_t A = smem_u32(base + (size_t)stage * sbytes);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = r0 + 32 * i;
          const int row = m_tile * kTileM + r;
          const bool ok = row < t.T && col < t.K;
          cp_async_16(A + (uint32_t)r * 128u + (((uint32_t)j ^ ((uint32_t)r & 7u)) << 4),
                      ok ? t.X + (size_t)row * t.K + col : t.X, ok ? 16u : 0u);
        }
        cp_async_mbar_arrive_noinc(&full[stage]);
        if (++stage == t.stages) { stage = 0; phase ^= 1u; }
      }
    } else {
      static_assert(kLoadDepth == 3, "the register ring below is written out for three slices");
      uint4 v0[4], v1[4], v2[4];
      issue(0, v0);
      issue(1, v1);
      for (int64_t g = 0; g < n_slices; g += 3) {
        issue(g + 2, v2);
        commit(g, v0);
        issue(g + 3, v0);
        commit(g + 1, v1);
        issue(g + 4, v1);
        commit(g + 2, v2);
      }
    }
  } else if (warp == kWWarp) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < my_items; ++it) {
        const int64_t item = first + it * stride;
        const int pass = (int)(item % t.n_pass);
        const int nb = (pass_rows(t.N, pass, t.pw) + 15) / 16 * 16;
        const uint32_t wbytes = (uint32_t)nb * 128u;
        const __half* src = t.img + pass_offset_halves(t.N, t.K, pass, t.pw);
        for (int ks = 0; ks < t.n_ks; ++ks) {
          mbar_wait(&empty[stage], phase ^ 1u);
          mbar_arrive_expect_tx(&full[stage], wbytes);
          bulk_g2s(base + (size_t)stage * sbytes + kABytes, src + (size_t)ks * nb * kSliceK, wbytes, &full[stage]);
          if (++stage == t.stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t it = 0; it < my_items; ++it) {
        const int64_t item = first + it * stride;
        const int pass = (int)(item % t.n_pass);
        const int nb = (pass_rows(t.N, pass, t.pw) + 15) / 16 * 16;
        const uint32_t idesc = make_idesc_f16(kTileM, nb);
        const int buf = (int)(it & 1);
        mbar_wait(&tmem_empty[buf], (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kMaxN);
        for (int ks = 0; ks < t.n_ks; ++ks) {
          mbar_wait(&full[stage], phase);
          fence_proxy_async();
          tc_fence_after();
          const uint32_t a_addr = smem_u32(base + (size_t)stage * sbytes);
          const uint64_t a_desc = make_kmajor_sw128_desc(a_addr);
          const uint64_t b_desc = make_kmajor_sw128_desc(a_addr + kABytes);
#pragma unroll
          for (int k = 0; k < kSliceK / 16; ++k)
            umma_f16(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (ks | k) != 0 ? 1u : 0u);
          umma_commit(&empty[stage]);
          if (++stage == t.stages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(&tmem_full[buf]);
      }
    }
  } else {
    // epilogue: TMEM -> + bias -> activation -> fp16 -> shared staging -> global.  A thread owns one token
    // row of the accumulator; the two warps of a lane quarter split the 32-column chunks (even / odd).
    // Storing straight from the row owner would issue 32 separate 16-byte requests per instruction
    // (one per row) -- the L2 request rate, not bytes, then bounds the kernel -- so a chunk is staged in
    // shared memory and written out with 4 lanes per row: 64 contiguous bytes per request.
    const int q = warp & 3, half = warp >> 2;
    unsigned char* stg = epi_stage + (size_t)warp * kEpiWarpBytes;
    for (int64_t it = 0; it < my_items; ++it) {
      const int64_t item = first + it * stride;
      const int m_tile = tile_of(item), pass = (int)(item % t.n_pass);
      const int nb = pass_rows(t.N, pass, t.pw);
      const int n0 = pass * t.pw;
      const int buf = (int)(it & 1);
      const int row_base = m_tile * kTileM + q * 32;
      mbar_wait(&tmem_full[buf], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kMaxN);
      // chunks half*32, half*32 + 64, ...  (the sibling warp on the same scheduler hides the TMEM latency)
      for (int c0 = half * 32; c0 < nb; c0 += 64) {
        uint32_t v[32];
        tmem_ld32_async(taddr0 + (uint32_t)c0, v);
        tmem_ld_wait(v);
        const float4* b4 = reinterpret_cast<const float4*>(t.bias + n0 + c0);   // n0, c0 multiples of 32
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          uint32_t packed[4];
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            const float4 bb = __ldg(b4 + 2 * jj + h2);
            const int e = 8 * jj + 4 * h2;
            float x0 = __uint_as_float(v[e]) + bb.x, x1 = __uint_as_float(v[e + 1]) + bb.y;
            float x2 = __uint_as_float(v[e + 2]) + bb.z, x3 = __uint_as_float(v[e + 3]) + bb.w;
            if (t.act == 1) { x0 = gelu_erf(x0); x1 = gelu_erf(x1); x2 = gelu_erf(x2); x3 = gelu_erf(x3); }
            packed[2 * h2] = pack_half2(x0, x1);
            packed[2 * h2 + 1] = pack_half2(x2, x3);
          }
          *reinterpret_cast<uint4*>(stg + (uint32_t)lane * kEpiPitch + (uint32_t)jj * 16u) =
              make_uint4(packed[0], packed[1], packed[2], packed[3]);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int rr = i * 8 + (lane >> 2), ch = lane & 3;
          const uint4 w = *reinterpret_cast<const uint4*>(stg + (uint32_t)rr * kEpiPitch + (uint32_t)ch * 16u);
          const int grow = row_base + rr;
          if (grow < t.T) *reinterpret_cast<uint4*>(t.Y + (size_t)grow * t.N + n0 + c0 + ch * 8) = w;
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---- tcgen05 linear layer, weights resident in shared memory, activations through a TMA tensor map ---------
// For K <= 384 and N % 192 == 0.  A CTA owns ONE 192-column pass of the output for the whole launch: it
// bulk-copies that pass of the pre-swizzled weight image (n_ks x 24 KB) into shared memory once and then
// walks token tiles.  Per 128-token tile only the activations move: one thread issues a 2-D
// cp.async.bulk.tensor (TMA tensor map over X[T, K], box 64 x 128, SWIZZLE_128B -- the layout the UMMA
// A descriptor expects; rows past T are zero-filled by the hardware) per K slice.  That takes the L2 -> SM
// traffic per tile from 288 KB (activations + a 256-column weight slice per tile) to 96 KB and frees the
// eight loader warps: twelve epilogue warps (three per TMEM lane quarter, two 32-column chunks each) now
// drain a 128 x 192 accumulator while the next tile's MMAs run into the other TMEM buffer.
// Pass width 192, three activation stages.  (kResN = 128 -- 96 KB of resident weights, SIX stages, a whole token
// tile of TMA loads in flight -- was measured and is slower: QKV 58.1 vs 61.5 us, but out-proj 24.7 vs 22.7 and
// FFN-up 105.4 vs 90.2: the deeper prefetch does not pay for re-reading the activations 1.5x as often.)
constexpr int kResEpiWarps = kResN == 128 ? 8 : 12;   // two 32-column chunks per warp either way
constexpr int kResProdWarp = kResEpiWarps;
constexpr int kResMmaWarp = kResEpiWarps + 1;
constexpr int kResThreads = (kResEpiWarps + 2) * 32;
constexpr int kResStages = kResN == 128 ? 6 : 3;
constexpr int kResChunkStride = (kResEpiWarps / 4) * 32;   // columns between a warp's two chunks
static_assert(kResN / 32 == 2 * (kResEpiWarps / 4), "two chunks per epilogue warp");
constexpr uint32_t kResWSliceBytes = kResN * 128u;                    // one K slice of the pass: 24 KB
constexpr uint32_t kResEpiBytes = kResEpiWarps * kEpiWarpBytes;

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__global__ void __launch_bounds__(kResThreads, 1) linear_wres_kernel(const __grid_constant__ CUtensorMap tmA, const LinArgs t) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  unsigned char* w_smem = base;                                               // [n_ks][192 x 128 B]
  unsigned char* a_smem = w_smem + (size_t)t.n_ks * kResWSliceBytes;          // [kResStages][16 KB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_smem + (size_t)kResStages * kABytes);
  uint64_t* a_full = bars;                   // [kResStages]
  uint64_t* a_empty = a_full + kResStages;   // [kResStages]
  uint64_t* tmem_full = a_empty + kResStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;         // [2]
  uint64_t* w_full = tmem_empty + 2;            // [1]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(w_full + 1);
  unsigned char* epi_stage = reinterpret_cast<unsigned char*>(bars) + kBarBytes;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = (t.T + kTileM - 1) / kTileM;
  // grid = n_pass * ctas_per_pass: CTA c serves pass c % n_pass and token tiles c / n_pass, + ctas_per_pass, ...
  const int pass = (int)(blockIdx.x % (unsigned)t.n_pass);
  const int first = (int)(blockIdx.x / (unsigned)t.n_pass), stride = (int)(gridDim.x / (unsigned)t.n_pass);
  const int my_items = first < m_tiles ? (m_tiles - first + stride - 1) / stride : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kResStages; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], kResEpiWarps);
    }
    mbar_init(w_full, 1);
    fence_barrier_init();
  }
  if (warp == kResMmaWarp) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == kResProdWarp) {
    if (lane == 0 && my_items > 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
      // the pass's weights: resident for the whole launch
      const __half* wsrc = t.img + pass_offset_halves(t.N, t.K, pass, kResN);
      mbar_arrive_expect_tx(w_full, (uint32_t)t.n_ks * kResWSliceBytes);
      for (int ks = 0; ks < t.n_ks; ++ks)
        bulk_g2s(w_smem + (size_t)ks * kResWSliceBytes, wsrc + (size_t)ks * kResN * kSliceK, kResWSliceBytes, w_full);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < my_items; ++it) {
        const int m_tile = first + it * stride;
        for (int ks = 0; ks < t.n_ks; ++ks) {
          mbar_wait(&a_empty[stage], phase ^ 1u);
          mbar_arrive_expect_tx(&a_full[stage], (uint32_t)kABytes);
          tma_load_2d(a_smem + (size_t)stage * kABytes, &tmA, ks * kSliceK, m_tile * kTileM, &a_full[stage]);
          if (++stage == kResStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == kResMmaWarp) {
    if (lane == 0 && my_items > 0) {
      const uint32_t idesc = make_idesc_f16(kTileM, kResN);
      mbar_wait(w_full, 0u);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < my_items; ++it) {
        const int buf = it & 1;
        mbar_wait(&tmem_empty[buf], (uint32_t)(((it >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kMaxN);
        for (int ks = 0; ks < t.n_ks; ++ks) {
          mbar_wait(&a_full[stage], phase);
          tc_fence_after();
          const uint64_t a_desc = make_kmajor_sw128_desc(smem_u32(a_smem + (size_t)stage * kABytes));
          const uint64_t b_desc = make_kmajor_sw128_desc(smem_u32(w_smem + (size_t)ks * kResWSliceBytes));
#pragma unroll
          for (int k = 0; k < kSliceK / 16; ++k)
            umma_f16(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (ks | k) != 0 ? 1u : 0u);
          umma_commit(&a_empty[stage]);
          if (++stage == kResStages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(&tmem_full[buf]);
      }
    }
  } else {
    // epilogue: warp w drains TMEM lane quarter w % 4 (hardware rule); the three warps of a quarter take the
    // 32-column chunks {i, i + 3} (i = w / 4).  Bias, activation, fp16, shared staging, 64-byte row stores.
    // The CTA's pass and each warp's two chunks never change, so the 64 bias values a thread needs live in
    // registers for the whole launch (ncu: with a bias load in front of every add, the epilogue warps spent a
    // third of their samples stalled on those loads and set the pace of the kernel).
    const int q = warp & 3, third = warp >> 2;
    unsigned char* stg = epi_stage + (size_t)warp * kEpiWarpBytes;
    const int n0 = pass * kResN;
    float bias_r[2][32];
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const float4* b4 = reinterpret_cast<const float4*>(t.bias + n0 + third * 32 + c * kResChunkStride);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float4 bb = __ldg(b4 + e);
        bias_r[c][4 * e] = bb.x; bias_r[c][4 * e + 1] = bb.y; bias_r[c][4 * e + 2] = bb.z; bias_r[c][4 * e + 3] = bb.w;
      }
    }
    for (int it = 0; it < my_items; ++it) {
      const int m_tile = first + it * stride;
      const int buf = it & 1;
      const int row_base = m_tile * kTileM + q * 32;
      mbar_wait(&tmem_full[buf], (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kMaxN);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const int c0 = third * 32 + c * kResChunkStride;
        uint32_t v[32];
        tmem_ld32_async(taddr0 + (uint32_t)c0, v);
        tmem_ld_wait(v);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          uint32_t packed[4];
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            const int e = 8 * jj + 4 * h2;
            float x0 = __uint_as_float(v[e]) + bias_r[c][e], x1 = __uint_as_float(v[e + 1]) + bias_r[c][e + 1];
            float x2 = __uint_as_float(v[e + 2]) + bias_r[c][e + 2], x3 = __uint_as_float(v[e + 3]) + bias_r[c][e + 3];
            if (t.act == 1) { x0 = gelu_erf(x0); x1 = gelu_erf(x1); x2 = gelu_erf(x2); x3 = gelu_erf(x3); }
            packed[2 * h2] = pack_half2(x0, x1);
            packed[2 * h2 + 1] = pack_half2(x2, x3);
          }
          *reinterpret_cast<uint4*>(stg + (uint32_t)lane * kEpiPitch + (uint32_t)jj * 16u) =
              make_uint4(packed[0], packed[1], packed[2], packed[3]);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int rr = i * 8 + (lane >> 2), ch = lane & 3;
          const uint4 w = *reinterpret_cast<const uint4*>(stg + (uint32_t)rr * kEpiPitch + (uint32_t)ch * 16u);
          const int grow = row_base + rr;
          if (grow < t.T) *reinterpret_cast<uint4*>(t.Y + (size_t)grow * t.N + n0 + c0 + ch * 8) = w;
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kResMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---- embeddings + LayerNorm: one warp per token ----------------------------------------------------------
// NC columns per lane: 16 for H <= 512 (MiniLM, H = 384), 24 for H <= 768 (BERT-base).
template <int NC>
__global__ void __launch_bounds__(256) embed_ln_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ type_ids,
                                                       const int32_t* __restrict__ pos_ids, const __half* __restrict__ word,
                                                       const __half* __restrict__ pos, const __half* __restrict__ type,
                                                       const float* __restrict__ g, const float* __restrict__ bta, float eps,
                                                       int T, int H, int vocab, int max_pos, int type_vocab,
                                                       __half* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int tok = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tok >= T) return;
  // ids are validated on the host (_xenc.py); the clamp only keeps a bad caller from reading out of bounds
  const __half* w = word + (size_t)min(max(ids[tok], 0), vocab - 1) * H;
  const __half* p = pos + (size_t)min(max(pos_ids[tok], 0), max_pos - 1) * H;
  const __half* ty = type + (size_t)min(max(type_ids[tok], 0), type_vocab - 1) * H;
  float x[NC];  // H <= 32 NC
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    const int c = lane + 32 * i;
    x[i] = c < H ? __half2float(w[c]) + __half2float(p[c]) + __half2float(ty[c]) : 0.f;
    s += x[i];
  }
  const float mean = warp_sum_f(s) / (float)H;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    const int c = lane + 32 * i;
    if (c < H) var += (x[i] - mean) * (x[i] - mean);
  }
  const float rstd = rsqrtf(warp_sum_f(var) / (float)H + eps);
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    const int c = lane + 32 * i;
    if (c < H) out[(size_t)tok * H + c] = __float2half_rn((x[i] - mean) * rstd * g[c] + bta[c]);
  }
}

// out = LayerNorm(x + res), one warp per token.  H % 128 == 0 (384 for MiniLM): a lane owns the columns
// lane * 4 + 128 i, so every load / store instruction of the warp covers 256 contiguous bytes (8-byte pieces);
// the first version moved 2 bytes per lane and instruction and ran at 3.5 TB/s.  NC columns per lane as in
// embed_ln_kernel: H <= 32 NC (VEC: NC / 4 pieces of 128 columns).
template <bool VEC, int NC>
__global__ void __launch_bounds__(256) add_ln_kernel(const __half* __restrict__ xin, const __half* __restrict__ res,
                                                     const float* __restrict__ g, const float* __restrict__ bta, float eps,
                                                     int T, int H, __half* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int tok = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (tok >= T) return;
  static_assert(NC % 4 == 0, "VEC pieces hold four columns per lane");
  constexpr int NP = NC / 4;   // 128-column pieces (VEC)
  float x[NC];   // H <= 32 NC
  float s = 0.f;
  if (VEC) {
    const uint2* xi = reinterpret_cast<const uint2*>(xin + (size_t)tok * H);
    const uint2* ri = reinterpret_cast<const uint2*>(res + (size_t)tok * H);
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      if (i * 128 < H) {
        const uint2 a = __ldg(xi + lane + 32 * i), r = __ldg(ri + lane + 32 * i);
        const float2 a0 = __half22float2(*reinterpret_cast<const __half2*>(&a.x)), a1 = __half22float2(*reinterpret_cast<const __half2*>(&a.y));
        const float2 r0 = __half22float2(*reinterpret_cast<const __half2*>(&r.x)), r1 = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
        x[4 * i] = a0.x + r0.x; x[4 * i + 1] = a0.y + r0.y; x[4 * i + 2] = a1.x + r1.x; x[4 * i + 3] = a1.y + r1.y;
        s += (x[4 * i] + x[4 * i + 1]) + (x[4 * i + 2] + x[4 * i + 3]);
      } else {
        x[4 * i] = x[4 * i + 1] = x[4 * i + 2] = x[4 * i + 3] = 0.f;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const int c = lane + 32 * i;
      x[i] = c < H ? __half2float(xin[(size_t)tok * H + c]) + __half2float(res[(size_t)tok * H + c]) : 0.f;
      s += x[i];
    }
  }
  const float mean = warp_sum_f(s) / (float)H;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < NC; ++i) {
    const int c = VEC ? (i >> 2) * 128 : lane + 32 * i;   // (VEC: all four values of a piece are in or out together)
    if (c < H) var += (x[i] - mean) * (x[i] - mean);
  }
  const float rstd = rsqrtf(warp_sum_f(var) / (float)H + eps);
  if (VEC) {
    uint2* oo = reinterpret_cast<uint2*>(out + (size_t)tok * H);
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      if (i * 128 < H) {
        const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + lane + 32 * i);
        const float4 bb = __ldg(reinterpret_cast<const float4*>(bta) + lane + 32 * i);
        uint2 o;
        o.x = pack_half2((x[4 * i] - mean) * rstd * gg.x + bb.x, (x[4 * i + 1] - mean) * rstd * gg.y + bb.y);
        o.y = pack_half2((x[4 * i + 2] - mean) * rstd * gg.z + bb.z, (x[4 * i + 3] - mean) * rstd * gg.w + bb.w);
        oo[lane + 32 * i] = o;
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const int c = lane + 32 * i;
      if (c < H) out[(size_t)tok * H + c] = __float2half_rn((x[i] - mean) * rstd * g[c] + bta[c]);
    }
  }
}

// ---- attention: one block per (sequence, head), flash-style on mma.sync tensor cores ---------------------
// qkv [T, 3H] (Q | K | V), ctx [T, H].  head_dim must be 32 (MiniLM-L12-H384: 12 heads x 32).
// K and V of the head sit in shared memory (80-byte row pitch: conflict-free ldmatrix); each warp
// owns 16-query blocks: S = Q K^T with m16n8k16 (fp16 in, fp32 acc), online softmax in the exp2
// domain, O += P V with P re-packed from the S accumulators as the A operand.
constexpr int kAttPitch = 40;  // halves

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}

__device__ __forceinline__ float ex2_approx(float x) {   // 2^x, one MUFU op; ex2(-inf) = +0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Sequence indices of a call sorted by length, longest first (counting sort over the lengths; equal lengths in any
// order).  One CTA, once per forward.
constexpr int kMaxSeqLenBins = 2048;
__global__ void __launch_bounds__(1024) seq_order_kernel(const int32_t* __restrict__ cu, int P, int32_t* __restrict__ order) {
  __shared__ int cnt[kMaxSeqLenBins + 1];
  for (int i = threadIdx.x; i <= kMaxSeqLenBins; i += blockDim.x) cnt[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < P; i += blockDim.x) atomicAdd(&cnt[min(cu[i + 1] - cu[i], kMaxSeqLenBins)], 1);
  __syncthreads();
  if (threadIdx.x == 0) {   // exclusive prefix from the longest bin down: cnt[L] becomes the first slot of length L
    int run = 0;
    for (int b = kMaxSeqLenBins; b >= 0; --b) { const int c = cnt[b]; cnt[b] = run; run += c; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < P; i += blockDim.x) order[atomicAdd(&cnt[min(cu[i + 1] - cu[i], kMaxSeqLenBins)], 1)] = i;
}

// Two 16-query tiles per warp and key block: the K / V fragments are fetched from shared memory once and feed both
// tiles' MMAs, and the two tiles' softmax chains (max -> ex2 -> sum -> pack) interleave.  ncu on the one-tile
// kernel showed no saturated pipe (ex2 32 %, HMMA 30 %, issue 37 %) with three CTAs = 12 warps per SM: the
// dependent chain of a single tile per warp, not a throughput limit, set the pace.
//
// Launch order: one CTA per (sequence, head), heads fastest, the sequences walked longest first (`order`, built once per call by
// seq_order_kernel).  A CTA's work grows with L^2 and the lengths of a call spread over an order of magnitude; in
// arrival order a long sequence that starts in the last wave leaves most SMs idle while it finishes.  Longest first
// the last wave holds the shortest sequences.  The last key block is 32 keys wide when no more than 32 are left.
__global__ void __launch_bounds__(128, 3) attention2_kernel(const __half* __restrict__ qkv, const int32_t* __restrict__ cu,
                                                         const int32_t* __restrict__ order, int H, int n_heads,
                                                         float scale_log2e, __half* __restrict__ ctx, int n_seq, int seq_fastest, int stage_async) {
  extern __shared__ __align__(16) unsigned char att_smem[];
  // CTA -> (sequence slot, head): heads fastest (the twelve CTAs of a sequence run together and read the same qkv rows).
  // The run-time seq_fastest / stage_async / null-order cases are what rl_xenc_score does not use; folding them away
  // costs this kernel 52 bytes of spills at its 168-register cap (three CTAs per SM), so they stay parameters.
  const int head = seq_fastest ? (int)(blockIdx.x / (unsigned)n_seq) : (int)(blockIdx.x % (unsigned)n_heads);
  const int slot = seq_fastest ? (int)(blockIdx.x % (unsigned)n_seq) : (int)(blockIdx.x / (unsigned)n_heads);
  const int seq = order != nullptr ? order[slot] : slot;
  const int t0 = cu[seq], L = cu[seq + 1] - t0;
  const int Lp = (L + 63) / 64 * 64;
  __half* Ks = reinterpret_cast<__half*>(att_smem);
  __half* Vs = Ks + (size_t)Lp * kAttPitch;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t ld = (size_t)3 * H;
  if (stage_async) {
    // K / V of the head: global -> shared memory with cp.async (16 bytes each, zero-filled past the sequence), no
    // registers in between; the first Q fragments are requested below while these copies are in flight.
#pragma unroll 4
    for (int idx = threadIdx.x; idx < Lp * 4; idx += blockDim.x) {
      const int j = idx >> 2, c = idx & 3;
      const __half* base = qkv + (size_t)(t0 + (j < L ? j : L - 1)) * ld + head * 32 + c * 8;
      const uint32_t nbytes = j < L ? 16u : 0u;
      cp_async_16(smem_u32(Ks + (size_t)j * kAttPitch + c * 8), base + H, nbytes);
      cp_async_16(smem_u32(Vs + (size_t)j * kAttPitch + c * 8), base + 2 * H, nbytes);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  } else {
#pragma unroll 4
    for (int idx = threadIdx.x; idx < Lp * 4; idx += blockDim.x) {
      const int j = idx >> 2, c = idx & 3;
      uint4 kv = make_uint4(0u, 0u, 0u, 0u), vv = kv;
      if (j < L) {
        const __half* base = qkv + (size_t)(t0 + j) * ld + head * 32 + c * 8;
        kv = __ldg(reinterpret_cast<const uint4*>(base + H));
        vv = __ldg(reinterpret_cast<const uint4*>(base + 2 * H));
      }
      *reinterpret_cast<uint4*>(Ks + (size_t)j * kAttPitch + c * 8) = kv;
      *reinterpret_cast<uint4*>(Vs + (size_t)j * kAttPitch + c * 8) = vv;
    }
  }
  const int r = lane >> 2, cp = (lane & 3) * 2;
  auto load_q = [&](int qb, uint32_t (&a)[2][4]) {   // A fragments of S = Q K^T for one 16-query tile (rows >= L read as zero)
    const int q0 = qb * 16 + r, q1 = q0 + 8;
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      const __half* p0 = qkv + (size_t)(t0 + q0) * ld + head * 32 + ks * 16 + cp;
      const __half* p1 = qkv + (size_t)(t0 + q1) * ld + head * 32 + ks * 16 + cp;
      a[ks][0] = q0 < L ? __ldg(reinterpret_cast<const uint32_t*>(p0)) : 0u;
      a[ks][1] = q1 < L ? __ldg(reinterpret_cast<const uint32_t*>(p1)) : 0u;
      a[ks][2] = q0 < L ? __ldg(reinterpret_cast<const uint32_t*>(p0 + 8)) : 0u;
      a[ks][3] = q1 < L ? __ldg(reinterpret_cast<const uint32_t*>(p1 + 8)) : 0u;
    }
  };
  // Q fragments of the warp's first pair of tiles: global loads that overlap the K / V staging above.
  uint32_t a[2][2][4];
  load_q(2 * warp, a[0]);
  load_q(2 * warp + 1, a[1]);
  if (stage_async) asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  for (int pb = warp; pb * 32 < L; pb += 4) {   // this warp's pair of tiles: queries [32 pb, 32 pb + 32)
    float m[2][2], l[2][2], O[2][4][4];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      m[t][0] = m[t][1] = -INFINITY;
      l[t][0] = l[t][1] = 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) O[t][i][e] = 0.f;
    }
    // One block of NKK k-steps (16 keys each) starting at key kb: NKK = 4 for a full 64-key block, 1..3 for the tail of
    // the sequence.  NKK is a compile-time constant so that every loop unrolls without guards (run-time guards inside
    // the unrolled body kept the compiler from interleaving the MMAs with the softmax: 134 -> 161 us per layer).
    auto block = [&](auto nkk_tag, int kb) {
      constexpr int NKK = decltype(nkk_tag)::value;
      constexpr int NJ = 2 * NKK;   // 8-key score tiles
      float S[2][NJ][4];
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        uint32_t b[4];
        ldsm_x4(b, Ks + (size_t)(kb + j * 8 + (lane & 7)) * kAttPitch + (lane >> 3) * 8);
#pragma unroll
        for (int t = 0; t < 2; ++t) {
#pragma unroll
          for (int e = 0; e < 4; ++e) S[t][j][e] = 0.f;
          mma16816(S[t][j], a[t][0], b[0], b[1]);
          mma16816(S[t][j], a[t][1], b[2], b[3]);
        }
      }
      if (kb + NJ * 8 > L) {   // only the last key block holds padding keys
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int j = 0; j < NJ; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e)
              if (kb + j * 8 + cp + (e & 1) >= L) S[t][j][e] = -INFINITY;
      }
      float mn[2][2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          mx0 = fmaxf(mx0, fmaxf(S[t][j][0], S[t][j][1]));
          mx1 = fmaxf(mx1, fmaxf(S[t][j][2], S[t][j][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        // finite: every block holds at least one valid key (kb < L)
        mn[t][0] = fmaxf(m[t][0], mx0 * scale_log2e);
        mn[t][1] = fmaxf(m[t][1], mx1 * scale_log2e);
        const float c0 = ex2_approx(m[t][0] - mn[t][0]), c1 = ex2_approx(m[t][1] - mn[t][1]);
        l[t][0] *= c0; l[t][1] *= c1;
#pragma unroll
        for (int i = 0; i < 4; ++i) { O[t][i][0] *= c0; O[t][i][1] *= c0; O[t][i][2] *= c1; O[t][i][3] *= c1; }
        m[t][0] = mn[t][0]; m[t][1] = mn[t][1];
      }
#pragma unroll
      for (int t = 0; t < 2; ++t)
#pragma unroll
        for (int j = 0; j < NJ; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float pexp = ex2_approx(fmaf(S[t][j][e], scale_log2e, e < 2 ? -mn[t][0] : -mn[t][1]));   // -inf -> 0
            S[t][j][e] = pexp;
            if (e < 2) l[t][0] += pexp; else l[t][1] += pexp;
          }
#pragma unroll
      for (int kk = 0; kk < NKK; ++kk) {
        uint32_t pa[2][4];
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          pa[t][0] = pack_half2(S[t][2 * kk][0], S[t][2 * kk][1]);
          pa[t][1] = pack_half2(S[t][2 * kk][2], S[t][2 * kk][3]);
          pa[t][2] = pack_half2(S[t][2 * kk + 1][0], S[t][2 * kk + 1][1]);
          pa[t][3] = pack_half2(S[t][2 * kk + 1][2], S[t][2 * kk + 1][3]);
        }
#pragma unroll
        for (int dn2 = 0; dn2 < 2; ++dn2) {
          uint32_t vb[4];
          ldsm_x4_trans(vb, Vs + (size_t)(kb + kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * kAttPitch +
                                (dn2 * 2 + (lane >> 4)) * 8);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            mma16816(O[t][dn2 * 2], pa[t], vb[0], vb[1]);
            mma16816(O[t][dn2 * 2 + 1], pa[t], vb[2], vb[3]);
          }
        }
      }
    };
    // 64-key blocks while more than 32 keys are left (the last of them may hold padding keys), then at most one
    // 32-key block: a 200-token sequence computes 224 keys instead of 256 (L is warp-uniform).
    int kb = 0;
    for (; L - kb > 32; kb += 64) block(std::integral_constant<int, 4>{}, kb);
    if (L - kb > 0) block(std::integral_constant<int, 2>{}, kb);
    if ((pb + 4) * 32 < L) {   // the next pair's Q fragments travel while this pair's output is normalised and stored
      load_q(2 * (pb + 4), a[0]);
      load_q(2 * (pb + 4) + 1, a[1]);
    }
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      float l0 = l[t][0], l1 = l[t][1];
      l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
      l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
      l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
      const float inv0 = 1.f / l0, inv1 = 1.f / l1;
      const int q0 = (2 * pb + t) * 16 + r, q1 = q0 + 8;
#pragma unroll
      for (int dn = 0; dn < 4; ++dn) {
        if (q0 < L) *reinterpret_cast<uint32_t*>(ctx + (size_t)(t0 + q0) * H + head * 32 + dn * 8 + cp) = pack_half2(O[t][dn][0] * inv0, O[t][dn][1] * inv0);
        if (q1 < L) *reinterpret_cast<uint32_t*>(ctx + (size_t)(t0 + q1) * H + head * 32 + dn * 8 + cp) = pack_half2(O[t][dn][2] * inv1, O[t][dn][3] * inv1);
      }
    }
  }
}

// ---- attention for head_dim 64 (BERT-base: 12 heads x 64) ------------------------------------------------
// Same math as attention2_kernel (m16n8k16 fp16 MMAs, fp32 accumulate, online softmax in the exp2 domain) and the same
// launch order (one CTA per (sequence, head), heads fastest, sequences longest first).  Two things differ, both forced
// by the wider head:
//   - One 16-query tile per warp.  O (32 registers), the Q fragments (16) and the scores of a 64-key block (32) fit the
//     168-register cap of three CTAs per SM; two tiles per warp would need 160 for these alone and spill.  (At four
//     CTAs per SM, a 128-register cap, ptxas spills 16 bytes.)
//   - K and V stream through shared memory in 64-key blocks, double-buffered with cp.async, instead of staying
//     resident: a whole 512-token head at a 144-byte pitch is 147 KB, one CTA per SM.  The ring is 36 KB whatever the
//     sequence length.
// The CTA walks its queries in passes of 64 (warp w owns queries [64 p + 16 w, + 16)) and streams the head's keys once
// per pass; the block stream runs across passes, so the next pass's first block loads while this pass ends.  The last
// block of a pass is 16, 32 or 64 keys wide (the fewest that cover the keys left).
constexpr int kAtt64Pitch = 72;    // halves per staged key row: 144 bytes, conflict-free ldmatrix
constexpr int kAtt64Keys = 64;     // keys per streamed block
constexpr int kAtt64StageHalves = 2 * kAtt64Keys * kAtt64Pitch;   // K rows, then V rows
constexpr int kAtt64Stages = 2;

__global__ void __launch_bounds__(128, 3) attention64_kernel(const __half* __restrict__ qkv, const int32_t* __restrict__ cu,
                                                          const int32_t* __restrict__ order, int H, int n_heads,
                                                          float scale_log2e, __half* __restrict__ ctx) {
  __shared__ __align__(16) __half kv_smem[kAtt64Stages * kAtt64StageHalves];   // 36 864 bytes
  const int head = (int)(blockIdx.x % (unsigned)n_heads);
  const int seq = order[blockIdx.x / (unsigned)n_heads];
  const int t0 = cu[seq], L = cu[seq + 1] - t0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t ld = (size_t)3 * H;
  const int n_kb = (L + kAtt64Keys - 1) / kAtt64Keys;   // key blocks per pass
  const int n_blocks = (L + 63) / 64 * n_kb;            // passes x key blocks
  // Block g -> stage g % 2: K and V rows of keys [64 (g % n_kb), + 64), zero-filled past the sequence.
  auto load_block = [&](int g) {
    const int kb = (g % n_kb) * kAtt64Keys;
    __half* Ks = kv_smem + (g & 1) * kAtt64StageHalves;
    __half* Vs = Ks + kAtt64Keys * kAtt64Pitch;
#pragma unroll
    for (int i = 0; i < 4; ++i) {   // 64 keys x 8 16-byte chunks of K and of V, 128 threads
      const int idx = threadIdx.x + 128 * i;
      const int j = idx >> 3, c = idx & 7;
      const int key = kb + j;
      const __half* src = qkv + (size_t)(t0 + (key < L ? key : L - 1)) * ld + head * 64 + c * 8;
      const uint32_t nbytes = key < L ? 16u : 0u;
      cp_async_16(smem_u32(Ks + j * kAtt64Pitch + c * 8), src + H, nbytes);
      cp_async_16(smem_u32(Vs + j * kAtt64Pitch + c * 8), src + 2 * H, nbytes);
    }
  };
  const int r = lane >> 2, cp = (lane & 3) * 2;
  uint32_t a[4][4];   // Q fragments of the warp's tile (rows >= L read as zero)
  float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f}, O[8][4];
  // One key block of NKK k-steps (16 keys each); NKK is a compile-time constant so that the loops unroll without guards.
  auto block = [&](auto nkk_tag, const __half* Ks, const __half* Vs, int kb) {
    constexpr int NKK = decltype(nkk_tag)::value;
    constexpr int NJ = 2 * NKK;   // 8-key score tiles
    float S[NJ][4];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      uint32_t b[4], b2[4];
      ldsm_x4(b, Ks + (j * 8 + (lane & 7)) * kAtt64Pitch + (lane >> 3) * 8);          // dims 0..31
      ldsm_x4(b2, Ks + (j * 8 + (lane & 7)) * kAtt64Pitch + 32 + (lane >> 3) * 8);    // dims 32..63
#pragma unroll
      for (int e = 0; e < 4; ++e) S[j][e] = 0.f;
      mma16816(S[j], a[0], b[0], b[1]);
      mma16816(S[j], a[1], b[2], b[3]);
      mma16816(S[j], a[2], b2[0], b2[1]);
      mma16816(S[j], a[3], b2[2], b2[3]);
    }
    if (kb + NJ * 8 > L) {   // only the last key block holds padding keys
#pragma unroll
      for (int j = 0; j < NJ; ++j)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (kb + j * 8 + cp + (e & 1) >= L) S[j][e] = -INFINITY;
    }
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      mx0 = fmaxf(mx0, fmaxf(S[j][0], S[j][1]));
      mx1 = fmaxf(mx1, fmaxf(S[j][2], S[j][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    // finite: every block holds at least one valid key (kb < L)
    const float mn0 = fmaxf(m[0], mx0 * scale_log2e), mn1 = fmaxf(m[1], mx1 * scale_log2e);
    const float c0 = ex2_approx(m[0] - mn0), c1 = ex2_approx(m[1] - mn1);
    l[0] *= c0; l[1] *= c1;
#pragma unroll
    for (int i = 0; i < 8; ++i) { O[i][0] *= c0; O[i][1] *= c0; O[i][2] *= c1; O[i][3] *= c1; }
    m[0] = mn0; m[1] = mn1;
#pragma unroll
    for (int j = 0; j < NJ; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float pexp = ex2_approx(fmaf(S[j][e], scale_log2e, e < 2 ? -mn0 : -mn1));   // -inf -> 0
        S[j][e] = pexp;
        if (e < 2) l[0] += pexp; else l[1] += pexp;
      }
#pragma unroll
    for (int kk = 0; kk < NKK; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_half2(S[2 * kk][0], S[2 * kk][1]);
      pa[1] = pack_half2(S[2 * kk][2], S[2 * kk][3]);
      pa[2] = pack_half2(S[2 * kk + 1][0], S[2 * kk + 1][1]);
      pa[3] = pack_half2(S[2 * kk + 1][2], S[2 * kk + 1][3]);
#pragma unroll
      for (int dn2 = 0; dn2 < 4; ++dn2) {
        uint32_t vb[4];
        ldsm_x4_trans(vb, Vs + (kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * kAtt64Pitch + (dn2 * 2 + (lane >> 4)) * 8);
        mma16816(O[dn2 * 2], pa, vb[0], vb[1]);
        mma16816(O[dn2 * 2 + 1], pa, vb[2], vb[3]);
      }
    }
  };
  if (n_blocks > 0) load_block(0);
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (int g = 0; g < n_blocks; ++g) {
    const int pass = g / n_kb, kbi = g - pass * n_kb, kb = kbi * kAtt64Keys;
    if (g + 1 < n_blocks) load_block(g + 1);
    asm volatile("cp.async.commit_group;" ::: "memory");   // (an empty group at the end keeps the wait below uniform)
    const int q0 = pass * 64 + warp * 16 + r, q1 = q0 + 8;
    const bool active = pass * 64 + warp * 16 < L;   // warp-uniform: the tile holds at least one query
    if (active && kbi == 0) {   // a new pass: this warp's Q fragments and a fresh softmax state
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const __half* p0 = qkv + (size_t)(t0 + q0) * ld + head * 64 + ks * 16 + cp;
        const __half* p1 = qkv + (size_t)(t0 + q1) * ld + head * 64 + ks * 16 + cp;
        a[ks][0] = q0 < L ? __ldg(reinterpret_cast<const uint32_t*>(p0)) : 0u;
        a[ks][1] = q1 < L ? __ldg(reinterpret_cast<const uint32_t*>(p1)) : 0u;
        a[ks][2] = q0 < L ? __ldg(reinterpret_cast<const uint32_t*>(p0 + 8)) : 0u;
        a[ks][3] = q1 < L ? __ldg(reinterpret_cast<const uint32_t*>(p1 + 8)) : 0u;
      }
      m[0] = m[1] = -INFINITY;
      l[0] = l[1] = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int e = 0; e < 4; ++e) O[i][e] = 0.f;
    }
    asm volatile("cp.async.wait_group 1;" ::: "memory");   // block g has landed (this thread's copies) ...
    __syncthreads();                                        // ... and every thread's
    if (active) {
      const __half* Ks = kv_smem + (g & 1) * kAtt64StageHalves;
      const __half* Vs = Ks + kAtt64Keys * kAtt64Pitch;
      const int rem = L - kb;
      if (rem > 32) block(std::integral_constant<int, 4>{}, Ks, Vs, kb);
      else if (rem > 16) block(std::integral_constant<int, 2>{}, Ks, Vs, kb);
      else block(std::integral_constant<int, 1>{}, Ks, Vs, kb);
      if (kbi == n_kb - 1) {   // the pass is done: normalise and store this warp's 16 rows
        float s0 = l[0], s1 = l[1];
        s0 += __shfl_xor_sync(0xffffffffu, s0, 1);
        s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
        s1 += __shfl_xor_sync(0xffffffffu, s1, 1);
        s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
        const float inv0 = 1.f / s0, inv1 = 1.f / s1;
#pragma unroll
        for (int dn = 0; dn < 8; ++dn) {
          if (q0 < L) *reinterpret_cast<uint32_t*>(ctx + (size_t)(t0 + q0) * H + head * 64 + dn * 8 + cp) = pack_half2(O[dn][0] * inv0, O[dn][1] * inv0);
          if (q1 < L) *reinterpret_cast<uint32_t*>(ctx + (size_t)(t0 + q1) * H + head * 64 + dn * 8 + cp) = pack_half2(O[dn][2] * inv1, O[dn][3] * inv1);
        }
      }
    }
    __syncthreads();   // stage g % 2 is free for block g + 2
  }
}

// ---- pooler + classifier ----------------------------------------------------------------------------------
// logit[s] = Wc . tanh(Wp h_s + bp) + bc with h_s the [CLS] row of sequence s.  A CTA owns kClsSeqs sequences
// (their [CLS] rows sit in shared memory as fp32) and its H/32 warps share the H pooler outputs; for one output
// the lanes stride over the H inputs, so every Wp read is a coalesced 128-byte line shared by the CTA's
// sequences, followed by one warp-shuffle reduction per sequence; the warps' partial logits meet in shared
// memory and are summed in a fixed order.  (History: Wp row-per-lane, 32 lines per load instruction: 313 us per
// launch; then one WARP per four sequences walking all H outputs one after the other: coalesced, but 16 CTAs of
// serial work, 526 us per 256-sequence call = 9 % of the forward in the round-2 launch list.)
constexpr int kClsSeqs = 2;
constexpr int kClsMaxWarps = 16;
__global__ void __launch_bounds__(kClsMaxWarps * 32) cls_head_kernel(const __half* __restrict__ hidden, const int32_t* __restrict__ cu,
                                                                     const float* __restrict__ Wp, const float* __restrict__ bp,
                                                                     const float* __restrict__ Wc, const float* __restrict__ bc,
                                                                     int P, int H, float* __restrict__ logit,
                                                                     float* __restrict__ score) {
  extern __shared__ float cls_smem[];  // [kClsSeqs][H] [CLS] rows as fp32, then [warps][kClsSeqs] partial logits
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int seq0 = blockIdx.x * kClsSeqs;
  float* h = cls_smem;
  float* part = cls_smem + (size_t)kClsSeqs * H;
#pragma unroll
  for (int s = 0; s < kClsSeqs; ++s) {
    const bool ok = seq0 + s < P;
    const __half* src = hidden + (size_t)cu[ok ? seq0 + s : seq0] * H;  // [CLS] token
    for (int c = threadIdx.x; c < H; c += blockDim.x) h[s * H + c] = ok ? __half2float(src[c]) : 0.f;
  }
  __syncthreads();
  float out[kClsSeqs];
#pragma unroll
  for (int s = 0; s < kClsSeqs; ++s) out[s] = 0.f;
#pragma unroll 2
  for (int o = warp; o < H; o += nw) {   // this warp's pooler outputs
    const float* w = Wp + (size_t)o * H;
    float a[kClsSeqs];
#pragma unroll
    for (int s = 0; s < kClsSeqs; ++s) a[s] = 0.f;
#pragma unroll 4
    for (int c = lane; c < H; c += 32) {
      const float wv = __ldg(w + c);
#pragma unroll
      for (int s = 0; s < kClsSeqs; ++s) a[s] = fmaf(wv, h[s * H + c], a[s]);
    }
    const float b = __ldg(bp + o), wc = __ldg(Wc + o);
#pragma unroll
    for (int s = 0; s < kClsSeqs; ++s) out[s] += tanhf(warp_sum_f(a[s]) + b) * wc;   // identical on every lane
  }
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kClsSeqs; ++s) part[warp * kClsSeqs + s] = out[s];
  }
  __syncthreads();
  if (threadIdx.x < kClsSeqs && seq0 + threadIdx.x < P) {   // fixed summation order: deterministic logits
    float v = bc[0];
    for (int wi = 0; wi < nw; ++wi) v += part[wi * kClsSeqs + threadIdx.x];
    logit[seq0 + threadIdx.x] = v;
    score[seq0 + threadIdx.x] = 1.f / (1.f + __expf(-v));  // FlashRank: sigmoid of the single logit
  }
}

}  // namespace
}  // namespace rl

using namespace rl;

extern "C" size_t rl_xenc_linear_image_bytes(int N, int K) {
  const int n_ks = (K + kSliceK - 1) / kSliceK;
  const int n_pad = (N + 15) / 16 * 16;
  const int pw = pass_width(N, K);
  return (size_t)((n_pad + pw - 1) / pw) * pw * n_ks * kSliceK * sizeof(__half);
}

extern "C" int rl_xenc_pack_linear(const float* W, int N, int K, void* image, void* stream) {
  RL_REQUIRE(W && image && N > 0 && K > 0, RL_EINVAL, "rl_xenc_pack_linear: bad arguments");
  RL_REQUIRE(N % 16 == 0 && K % 8 == 0, RL_EUNSUPPORTED, "rl_xenc_pack_linear: N %% 16 and K %% 8 must be 0");
  RL_CUDA_CHECK(cudaMemsetAsync(image, 0, rl_xenc_linear_image_bytes(N, K), (cudaStream_t)stream));
  pack_linear_kernel<<<1024, 256, 0, (cudaStream_t)stream>>>(W, N, K, pass_width(N, K), reinterpret_cast<__half*>(image));
  RL_CUDA_CHECK(cudaGetLastError());
  return RL_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

static int launch_linear_resident(const __half* X, const void* img, const float* bias, __half* Y, int T, int N, int K, int act,
                                  int sm_count, cudaStream_t stream) {
  EncodeTiledFn enc = encode_tiled_fn();
  RL_REQUIRE(enc != nullptr, RL_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
  RL_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15) == 0 && (K * 2) % 16 == 0, RL_EINVAL, "resident linear: X must be 16-byte aligned");
  CUtensorMap tm;
  const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)T};          // innermost first
  const cuuint64_t gstr[1] = {(cuuint64_t)K * sizeof(__half)};        // bytes between token rows
  const cuuint32_t box[2] = {(cuuint32_t)kSliceK, (cuuint32_t)kTileM};   // 64 halves (128 B, one swizzle row) x 128 tokens
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(X), gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RL_REQUIRE(r == CUDA_SUCCESS, RL_ECUDA, "cuTensorMapEncodeTiled failed (%d) for X[%d, %d]", (int)r, T, K);
  LinArgs t;
  t.X = X; t.img = reinterpret_cast<const __half*>(img); t.bias = bias; t.Y = Y; t.T = T; t.N = N; t.K = K; t.act = act;
  t.n_pass = N / kResN;
  t.n_ks = K / kSliceK;
  t.stages = kResStages;
  t.cp_async = 0;
  t.pw = kResN;
  const size_t smem = (size_t)t.n_ks * kResWSliceBytes + (size_t)kResStages * kABytes + kBarBytes + kResEpiBytes + 1024;
  RL_REQUIRE(smem <= 227 * 1024, RL_EUNSUPPORTED, "resident linear: %zu bytes of shared memory", smem);
  RL_CUDA_CHECK(cudaFuncSetAttribute(linear_wres_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int m_tiles = (T + kTileM - 1) / kTileM;
  int per_pass = sm_count / t.n_pass;
  if (per_pass < 1) per_pass = 1;
  if (per_pass > m_tiles) per_pass = m_tiles;
  linear_wres_kernel<<<t.n_pass * per_pass, kResThreads, smem, stream>>>(tm, t);
  RL_CUDA_CHECK(cudaGetLastError());
  return RL_OK;
}

static int launch_linear(const __half* X, const void* img, const float* bias, __half* Y, int T, int N, int K, int act,
                         int sm_count, cudaStream_t stream) {
  if (use_resident(N, K)) return launch_linear_resident(X, img, bias, Y, T, N, K, act, sm_count, stream);
  LinArgs t;
  t.X = X; t.img = reinterpret_cast<const __half*>(img); t.bias = bias; t.Y = Y; t.T = T; t.N = N; t.K = K; t.act = act;
  t.pw = pass_width(N, K);
  t.n_pass = (N + t.pw - 1) / t.pw;
  t.n_ks = (K + kSliceK - 1) / kSliceK;
  // The cp.async loader is the one used.  The register-ring branch stays in the kernel because the kernel with it
  // folded away measured slower on B200 (FFN-down, K = 1536: 95.5 vs 92.5 us, tools/time_linear.py).
  t.cp_async = 1;
  static_assert((2 * kMaxStages + 4) * 8 + 8 <= kBarBytes, "barrier block overflows its slot");
  const uint32_t tail = kBarBytes + kEpiBytes;
  int stages = (int)((kSmemBudget - 1024 - tail) / lin_stage_bytes());
  if (stages > kMaxStages) stages = kMaxStages;
  t.stages = stages;
  const size_t smem = (size_t)stages * lin_stage_bytes() + tail + 1024;
  RL_CUDA_CHECK(cudaFuncSetAttribute(linear_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t items = (int64_t)((T + kTileM - 1) / kTileM) * t.n_pass;
  const int grid = (int)(items < sm_count ? items : sm_count);
  linear_tcgen05_kernel<<<grid, kThreads, smem, stream>>>(t);
  RL_CUDA_CHECK(cudaGetLastError());
  return RL_OK;
}

extern "C" int rl_xenc_linear(const void* X, const void* image, const float* bias, void* Y, int T, int N, int K, int act,
                              void* stream) {
  RL_REQUIRE(X && image && bias && Y && T >= 0, RL_EINVAL, "rl_xenc_linear: bad arguments");
  RL_REQUIRE(N % 32 == 0 && K % 8 == 0, RL_EUNSUPPORTED, "rl_xenc_linear: N %% 32 and K %% 8 must be 0");
  RL_REQUIRE((reinterpret_cast<uintptr_t>(bias) & 15) == 0, RL_EINVAL, "rl_xenc_linear: bias must be 16-byte aligned");
  if (T == 0) return RL_OK;
  int dev = 0, sms = 148;
  RL_CUDA_CHECK(cudaGetDevice(&dev));
  RL_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  return launch_linear(reinterpret_cast<const __half*>(X), image, bias, reinterpret_cast<__half*>(Y), T, N, K, act, sms,
                       (cudaStream_t)stream);
}

extern "C" size_t rl_xenc_workspace_bytes(const rl_xenc_weights* w, int T) {
  if (w == nullptr || T < 0) return 0;
  const size_t H = (size_t)w->hidden, F = (size_t)w->ffn;
  // hidden, qkv (3H), ctx, tmp (H), ffn (F) -- fp16 rows
  // + the length-sorted sequence order of the call (at most T sequences), 16-byte aligned behind the rows
  return ((size_t)T * (H + 3 * H + H + H + F) * sizeof(__half) + (size_t)T * sizeof(int32_t) + 4096);
}

extern "C" int rl_xenc_score(const rl_xenc_weights* w, const int32_t* input_ids, const int32_t* type_ids,
                             const int32_t* pos_ids, const int32_t* cu_seqlens, int P, int T, int max_len,
                             float* out_logit, float* out_score, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  RL_REQUIRE(w && w->layers && input_ids && type_ids && pos_ids && cu_seqlens && out_logit && out_score, RL_EINVAL,
             "rl_xenc_score: null pointer");
  if (P == 0 || T == 0) return RL_OK;
  const int H = w->hidden, F = w->ffn, nh = w->n_heads;
  const int head_dim = nh > 0 && H % nh == 0 ? H / nh : 0;
  RL_REQUIRE(H % 32 == 0 && H > 0 && H <= 768 && (head_dim == 32 || head_dim == 64), RL_EUNSUPPORTED,
             "rl_xenc_score: hidden=%d heads=%d unsupported (supported: head_dim 32 or 64, hidden a multiple of 32 up to 768)",
             H, nh);
  RL_REQUIRE(F % 32 == 0 && max_len > 0 && max_len <= w->max_pos, RL_EUNSUPPORTED, "rl_xenc_score: bad ffn / max_len");
  RL_REQUIRE(workspace && workspace_bytes >= rl_xenc_workspace_bytes(w, T), RL_ENOSPACE, "rl_xenc_score: workspace too small");
  int dev = 0, sms = 148;
  RL_CUDA_CHECK(cudaGetDevice(&dev));
  RL_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  __half* hidden = reinterpret_cast<__half*>(workspace);
  __half* qkv = hidden + (size_t)T * H;
  __half* ctx = qkv + (size_t)T * 3 * H;
  __half* tmp = ctx + (size_t)T * H;
  __half* ffn = tmp + (size_t)T * H;
  int32_t* seq_order = reinterpret_cast<int32_t*>(
      (reinterpret_cast<uintptr_t>(ffn + (size_t)T * F) + 15) & ~uintptr_t(15));   // [P] (P <= T)
  RL_REQUIRE(P <= T, RL_EINVAL, "rl_xenc_score: more sequences than tokens");
  // Attention walks the sequences longest first.
  seq_order_kernel<<<1, 1024, 0, stream>>>(cu_seqlens, P, seq_order);
  RL_CUDA_CHECK(cudaGetLastError());
  const int tok_blocks = (T + 7) / 8;
  const bool ln_vec = H % 128 == 0;   // (LayerNorm gamma / beta come from torch allocations: 16-byte aligned)
  const bool ln_wide = H > 512;       // 24 columns per lane instead of 16
  const __half* word_emb = reinterpret_cast<const __half*>(w->word_emb);
  const __half* pos_emb = reinterpret_cast<const __half*>(w->pos_emb);
  const __half* type_emb = reinterpret_cast<const __half*>(w->type_emb);
  if (ln_wide)
    embed_ln_kernel<24><<<tok_blocks, 256, 0, stream>>>(input_ids, type_ids, pos_ids, word_emb, pos_emb, type_emb, w->emb_ln_g,
                                                        w->emb_ln_b, w->ln_eps, T, H, w->vocab, w->max_pos, w->type_vocab, hidden);
  else
    embed_ln_kernel<16><<<tok_blocks, 256, 0, stream>>>(input_ids, type_ids, pos_ids, word_emb, pos_emb, type_emb, w->emb_ln_g,
                                                        w->emb_ln_b, w->ln_eps, T, H, w->vocab, w->max_pos, w->type_vocab, hidden);
  RL_CUDA_CHECK(cudaGetLastError());
  auto add_ln = [&](const float* g, const float* b) {   // hidden = LayerNorm(tmp + hidden)
    if (ln_wide && ln_vec) add_ln_kernel<true, 24><<<tok_blocks, 256, 0, stream>>>(tmp, hidden, g, b, w->ln_eps, T, H, hidden);
    else if (ln_wide) add_ln_kernel<false, 24><<<tok_blocks, 256, 0, stream>>>(tmp, hidden, g, b, w->ln_eps, T, H, hidden);
    else if (ln_vec) add_ln_kernel<true, 16><<<tok_blocks, 256, 0, stream>>>(tmp, hidden, g, b, w->ln_eps, T, H, hidden);
    else add_ln_kernel<false, 16><<<tok_blocks, 256, 0, stream>>>(tmp, hidden, g, b, w->ln_eps, T, H, hidden);
  };
  size_t att_smem = 0;
  if (head_dim == 32) {   // attention2_kernel stages the whole head; attention64_kernel streams it (static 36 KB)
    att_smem = (size_t)((max_len + 63) / 64 * 64) * kAttPitch * 2 * sizeof(__half);
    RL_REQUIRE(att_smem <= 200 * 1024, RL_EUNSUPPORTED, "rl_xenc_score: max_len=%d too long for the attention kernel", max_len);
    RL_CUDA_CHECK(cudaFuncSetAttribute(attention2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem));
  }
  const float scale = 1.4426950408889634f / sqrtf((float)head_dim);  // softmax in the exp2 domain
  for (int l = 0; l < w->n_layers; ++l) {
    const rl_xenc_layer& L = w->layers[l];
    int rc = launch_linear(hidden, L.qkv_img, L.qkv_bias, qkv, T, 3 * H, H, 0, sms, stream);
    if (rc != RL_OK) return rc;
    if (head_dim == 32)
      attention2_kernel<<<(unsigned)P * (unsigned)nh, 128, att_smem, stream>>>(qkv, cu_seqlens, seq_order, H, nh, scale, ctx,
                                                                              P, /*seq_fastest=*/0, /*stage_async=*/1);
    else
      attention64_kernel<<<(unsigned)P * (unsigned)nh, 128, 0, stream>>>(qkv, cu_seqlens, seq_order, H, nh, scale, ctx);
    RL_CUDA_CHECK(cudaGetLastError());
    rc = launch_linear(ctx, L.o_img, L.o_bias, tmp, T, H, H, 0, sms, stream);
    if (rc != RL_OK) return rc;
    add_ln(L.ln1_g, L.ln1_b);
    RL_CUDA_CHECK(cudaGetLastError());
    rc = launch_linear(hidden, L.up_img, L.up_bias, ffn, T, F, H, 1, sms, stream);
    if (rc != RL_OK) return rc;
    rc = launch_linear(ffn, L.down_img, L.down_bias, tmp, T, H, F, 0, sms, stream);
    if (rc != RL_OK) return rc;
    add_ln(L.ln2_g, L.ln2_b);
    RL_CUDA_CHECK(cudaGetLastError());
  }
  const int cls_warps = H / 32 < kClsMaxWarps ? H / 32 : kClsMaxWarps;
  cls_head_kernel<<<(P + kClsSeqs - 1) / kClsSeqs, cls_warps * 32, ((size_t)kClsSeqs * H + kClsMaxWarps * kClsSeqs) * sizeof(float), stream>>>(
      hidden, cu_seqlens, w->pooler_w, w->pooler_b, w->cls_w, w->cls_b, P, H, out_logit, out_score);
  RL_CUDA_CHECK(cudaGetLastError());
  return RL_OK;
}
