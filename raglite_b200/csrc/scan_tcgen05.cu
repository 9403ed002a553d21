// tcgen05 / TMEM scan (RL_ALGO_TCGEN05) for sm_100a.
//
// Replaces the per-row distance expression DuckDB evaluates for vector_search (reference
// _search.py:69-79, _typing.py:123-134) with a coarse tensor-core pass whose survivors are
// re-scored exactly in float64 by the finalize kernel (select_finalize.cu).
//
// One persistent CTA per SM walks its tiles of 128 corpus rows:
//   * 8 loader warps stream the fp32 rows from HBM with coalesced 128-bit loads, scale them (cosine:
//     1/|e|, dot/l2: a global power of two), round to fp16 and store them into a 128B-swizzled
//     K-major shared-memory tile (the UMMA A operand),
//   * one thread bulk-copies (cp.async.bulk, the TMA engine) the matching 64-wide K slice of the
//     pre-swizzled fp16 query image (the UMMA B operand, N = #queries <= 256),
//   * one thread issues tcgen05.mma (M=128, N=#queries, K=16, fp32 accumulate in TMEM); two
//     accumulator buffers in TMEM let the epilogue of tile i overlap the MMAs of tile i+1,
//   * 4 epilogue warps read the accumulators with tcgen05.ld (lane = corpus row, column = query),
//     turn them into keys and either dump them (sample tiles) or compare them with the per-query
//     threshold; the few survivors are staged in shared memory together with a histogram of their
//     keys, flushed in bulk (one global atomic per touched query / bin), and the global histogram is
//     read back to tighten the thresholds while the scan is running (online refinement).
// All hand-offs are mbarrier based (full/empty per smem stage, full/empty per TMEM buffer).
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "scan_tcgen05.cuh"
#include "tcgen05_ptx.cuh"

namespace rl {

namespace {

using namespace tc;

constexpr int kTileM = 128;           // corpus rows per tile (UMMA M)
constexpr int kSliceK = 64;           // fp16 elements per K slice = one 128-byte swizzle row
constexpr int kMaxQ = 256;            // queries per pass (UMMA N <= 256)
constexpr int kNumEpiWarps = 4;       // warps 0..3 (TMEM lane quarter == warp index)
constexpr int kMmaWarp = 4;
constexpr int kQWarp = 5;
constexpr int kFirstLoaderWarp = 6;
constexpr int kNumLoaderWarps = 8;
constexpr int kThreads = (kFirstLoaderWarp + kNumLoaderWarps) * 32;  // 448
constexpr int kMaxStages = 8;
constexpr int kABytes = kTileM * 128;  // 16 KB per stage
constexpr uint32_t kSmemBudget = 222 * 1024;
constexpr int kPrefetchItems = 6;      // L2 prefetch distance in K-slice items (6 x 32 KB per SM)
constexpr int kPrefetchPairs = kPrefetchItems / 2;   // the same distance for the fast fp32 loader, in pairs of items
constexpr int kListCap = 1024;         // staged hit records (12 KB)
constexpr int kFlushFirst = 192;       // first flush early: it feeds the histogram that tightens the thresholds
constexpr int kFlushAt = 512;          // later flushes: once this many hits are waiting (or at the end)
constexpr int kRefreshEvery = 16;      // tiles between threshold refreshes from the global histogram
         // staged hit records per tile before falling back to direct emits

struct TcArgs {
  ScanArgs a;
  const __half* qimg;     // [n_ks][nq][64] fp16, rows pre-swizzled
  const float* q_scale;   // [B] key = acc * q_scale[b] (+ bias)
  const float* row_stats; // [2] max norm, max |element|
  int nq;                 // padded #queries of a FULL group (multiple of 16; kMaxQ when par_groups > 1)
  int nq_last;            // padded #queries of the last group
  int par_groups;         // > 1: group-parallel -- CTA c serves query group c % par_groups of the tiles of lane c / par_groups
  int n_ks;               // K slices
  int stages;
  int tmem_cols;          // allocated TMEM columns (power of two >= 2 * buf_cols)
  int buf_cols;           // columns per accumulator buffer (nq rounded up to 32)
  int tma_rows;           // fp16 storage: 1 = corpus tiles come through the tensor map (no loader warps)
};

// TMA tensor-map tile load (2-D, 128B swizzle: the UMMA K-major SW128 layout) and its L2-only prefetch.
__device__ __forceinline__ void tma_load_tile(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_tile(const CUtensorMap* tmap, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(tmap), "r"(c0), "r"(c1) : "memory");
}

// Global power-of-two row scale for the dot / l2 metrics (keeps |x| <= 1 in fp16).
__device__ __forceinline__ float pow2_scale(float max_abs) {
  return max_abs > 0.f ? exp2f(-ceilf(log2f(max_abs))) : 1.f;
}

struct SmemLayout {
  unsigned char* stage_base;  // stages * (kABytes + nq*128)
  uint64_t* full;             // [kMaxStages]
  uint64_t* empty;            // [kMaxStages]
  uint64_t* tmem_full;        // [2]
  uint64_t* tmem_empty;       // [2]
  uint32_t* tmem_ptr;
  float* thr;                 // [kMaxQ]
  float* cs;                  // [kMaxQ]
  float* thr0;                // [kMaxQ] threshold from the sample (histogram origin)
  float* inv_w;               // [kMaxQ] 1 / bin width (bin width = 4 eps)
  uint32_t* hist;             // [kMaxQ * kHistBins / 2] staged histogram, two 16-bit counters per word
  int* cnt;                   // [kMaxQ] hits per query staged since the last flush
  int* basev;                 // [kMaxQ] global slot base per query for the current flush
  int* list_n;                // [2] number of staged records (ping-pong by tile parity)
  uint32_t* list;             // [kListCap][3] {col | rank << 16, key bits, row}
};

__host__ __device__ inline uint32_t stage_bytes(int nq) { return kABytes + (uint32_t)nq * 128u; }
// Per query of the CTA's group: threshold, scale, histogram origin / bin width, the staged histogram and the
// counters, all in shared memory.
__host__ __device__ inline uint32_t tail_bytes() {
  const uint32_t per_q = 6u * 4u + (uint32_t)kHistBins * 2u;
  return (2 * kMaxStages + 4) * 8 + 16 + kMaxQ * per_q + 16 + kListCap * 12;
}

// PAIR: two CTAs of a cluster (an SM pair) issue one cta_group::2 MMA (M = 256: 128 rows per CTA) and
// each holds only half of the queries in shared memory, which halves the L2 -> SM query stream.
// EF16: the corpus is stored as fp16 (lossless for RAGLite data, whose embeddings are fp16-rounded,
// reference _embed.py:140): rows are copied into the swizzled tile without conversion, half the HBM bytes.
template <int METRIC, bool PAIR, bool EF16>
__global__ void __maxnreg__(128) scan_tcgen05_kernel(const __grid_constant__ CUtensorMap tmE, const TcArgs t) {
  extern __shared__ unsigned char smem_dyn[];
  // Group-parallel mode (B > 256): the CTAs of a "lane" -- par_groups consecutive CTAs -- walk the SAME corpus
  // tiles at the same time, one 256-query group each.  The first of them pulls a tile in from HBM, the others
  // find it in L2 microseconds later, so HBM sees the corpus once.
  const int P = t.par_groups > 1 ? t.par_groups : 1;
  const int pg = P > 1 ? (int)((PAIR ? blockIdx.x >> 1 : blockIdx.x) % (unsigned)P) : 0;
  ScanArgs a = t.a;
  const float* q_scale_g = t.q_scale;
  const __half* qimg_g = t.qimg;
  int nq = t.nq;                         // padded width of the group this CTA serves
  if (P > 1) {
    const int q0p = pg * kMaxQ;
    a.B = min(kMaxQ, t.a.B - q0p);
    a.thr += q0p; a.cand_cnt += q0p; a.eps += q0p; a.hist_inv_w += q0p; a.q_inv_norm += q0p;
    if (a.cnt_all != nullptr) a.cnt_all += q0p;
    a.dump += (size_t)q0p * a.n_sample_rows;
    a.cand += (size_t)q0p * a.cap;
    a.ghist += (size_t)q0p * kHistBins;
    q_scale_g += q0p;
    qimg_g += (size_t)pg * t.n_ks * kMaxQ * kSliceK;
    nq = (pg == P - 1) ? t.nq_last : t.nq;
  }
  // 1024-byte alignment for the 128B-swizzled tiles.
  // (pointer arithmetic on the __shared__ array keeps the address space known: LDS/STS, not generic LD/ST)
  unsigned char* base = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const uint32_t sbytes = stage_bytes(PAIR ? t.nq / 2 : t.nq);   // sized by a full group
  SmemLayout s;
  s.stage_base = base;
  s.full = reinterpret_cast<uint64_t*>(base + (size_t)t.stages * sbytes);
  s.empty = s.full + kMaxStages;
  s.tmem_full = s.empty + kMaxStages;
  s.tmem_empty = s.tmem_full + 2;
  s.tmem_ptr = reinterpret_cast<uint32_t*>(s.tmem_empty + 2);
  // Per-query arrays.  Their pitch goes through an opaque move: with compile-time offsets ptxas keeps one pointer
  // per array live across every warp role, and the dot / l2 instantiations spill at the 128-register cap.
  int qp = kMaxQ;
  asm volatile("" : "+r"(qp));
  s.thr = reinterpret_cast<float*>(s.tmem_ptr + 4);
  s.cs = s.thr + qp;
  s.thr0 = s.cs + qp;
  s.inv_w = s.thr0 + qp;
  s.hist = reinterpret_cast<uint32_t*>(s.inv_w + qp);
  s.cnt = reinterpret_cast<int*>(s.hist + qp * kHistBins / 2);
  s.basev = s.cnt + qp;
  s.list_n = s.basev + qp;
  s.list = reinterpret_cast<uint32_t*>(s.list_n + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Work units: blocks of 128 rows (single CTA) or pairs of consecutive block ordinals (PAIR: CTA
  // `rank` of the cluster takes ordinal 2 * unit + rank; a missing second block is an empty tile).
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const int64_t n_tiles = PAIR ? (a.n_mode_blocks + 1) / 2 : a.n_mode_blocks;
  const int64_t first = (PAIR ? (int64_t)(blockIdx.x >> 1) : (int64_t)blockIdx.x) / P;
  const int64_t stride = (PAIR ? (int64_t)(gridDim.x >> 1) : (int64_t)gridDim.x) / P;
  const int64_t my_tiles = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;
  auto ord_of = [&](int64_t tile) -> int64_t {
    const int64_t unit = first + tile * stride;
    return PAIR ? 2 * unit + rank : unit;
  };

  if (threadIdx.x == 0) {
    for (int i = 0; i < t.stages; ++i) {
      // 8 loader warps + the query producer (expect_tx) [+ the peer CTA's relay in the leader]
      // loader warps (none when the tensor map brings the rows) + the producer (expect_tx) [+ the peer's relay]
      mbar_init(&s.full[i], ((EF16 && t.tma_rows) ? 0 : kNumLoaderWarps) + 1 + ((PAIR && rank == 0) ? 1 : 0));
      mbar_init(&s.empty[i], 1);                   // one tcgen05.commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s.tmem_full[i], 1);
      mbar_init(&s.tmem_empty[i], PAIR ? 2 * kNumEpiWarps : kNumEpiWarps);  // PAIR: both CTAs' epilogues
    }
    fence_barrier_init();
  }
  for (int i = threadIdx.x; i < kMaxQ; i += blockDim.x) {
    s.thr[i] = (i < a.B && !a.dump_mode) ? a.thr[i] : __int_as_float(0x7f800000);  // +inf: never emit
    s.cs[i] = (i < a.B) ? q_scale_g[i] : 0.f;
    s.cnt[i] = 0;
    s.thr0[i] = s.thr[i];
    s.inv_w[i] = (i < a.B && !a.dump_mode) ? a.hist_inv_w[i] : 0.f;
  }
  for (int i = threadIdx.x; i < kMaxQ * kHistBins / 2; i += blockDim.x) s.hist[i] = 0u;
  if (threadIdx.x == 0) { s.list_n[0] = 0; s.list_n[1] = 0; }
  if (warp == kMmaWarp) {
    if (PAIR) tmem_alloc_2cta(s.tmem_ptr, (uint32_t)t.tmem_cols);
    else tmem_alloc(s.tmem_ptr, (uint32_t)t.tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // barriers of both CTAs are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *s.tmem_ptr;
  // Cosine on a corpus whose rows all have norm >= 0.5 and moderate magnitudes (the normal case:
  // embeddings are stored normalised): rows go to fp16 unscaled and the epilogue applies 1/|e|.
  const bool cos_noscale = METRIC == RL_METRIC_COSINE &&
                           (EF16 || (t.row_stats[2] > 0.f && t.row_stats[2] <= 2.f && t.row_stats[1] <= 1024.f &&
                                     t.row_stats[3] == 0.f));   // (the host only allows fp16 storage when this holds)

  // fp32 loader fast path (uniform): whole K slices in pairs, one query group per CTA, no per-row scale in the loader
  const bool fast_f32 = !EF16 && a.d % kSliceK == 0 && (t.n_ks & 1) == 0 && a.ld * 64 < (int64_t(1) << 32) &&
                        (METRIC != RL_METRIC_COSINE || cos_noscale);
  if (EF16 && t.tma_rows && warp >= kFirstLoaderWarp) {
    // fp16 storage through the tensor map: the producer thread issues one cp.async.bulk.tensor per K slice and the
    // TMA engine writes the 128B-swizzled tile itself -- these eight warps have nothing to do.
  } else if (EF16 && warp >= kFirstLoaderWarp) {
    // ===== corpus loaders, fp16 storage: HBM -> registers -> swizzled smem, no conversion =====
    // A K slice of a row is 128 bytes = 8 chunks of 16 bytes; thread lt owns chunk lt & 7 of rows
    // (lt >> 3) + 32 i.  Four items (4 x 16 KB per SM) stay in flight in registers.
    const int lt = threadIdx.x - kFirstLoaderWarp * 32;
    const int j = lt & 7, r0 = lt >> 3;
    const __half* Eh = reinterpret_cast<const __half*>(a.E);
    // (fp16-stored rows are used as they are: no global power-of-two scale -- it only guards the fp32 -> fp16
    // conversion against overflow -- and the query scale is built without it, see query_image_kernel)
    const int64_t total_items = my_tiles * t.n_ks;
    const size_t pitch32_bytes = (size_t)a.ld * 32 * sizeof(__half);
    const size_t slice_bytes = kSliceK * sizeof(__half);
    uint4 ring[4][4];
    int64_t ld_tile = 0;
    int ld_ks = 0, ld_rows = 0;
    const unsigned char* ld_ptr = nullptr;
    auto ld_set_tile = [&]() {
      if (ld_tile < my_tiles && ord_of(ld_tile) < a.n_mode_blocks) {
        const int64_t blk = mode_block_index(a, ord_of(ld_tile));
        const int64_t rem = a.n_rows - blk * kTileM;
        ld_rows = rem < kTileM ? (int)rem : kTileM;
        ld_ptr = reinterpret_cast<const unsigned char*>(Eh + (size_t)(blk * kTileM + r0) * a.ld + j * 8);
      } else {
        ld_rows = 0;
      }
    };
    int64_t pf_tile = 0;
    int pf_ks = 0, pf_rows = 0;
    const unsigned char* pf_ptr = nullptr;
    auto pf_set_tile = [&]() {   // only the first group's CTA of a lane prefetches
      if (pg == 0 && pf_tile < my_tiles && ord_of(pf_tile) < a.n_mode_blocks) {
        const int64_t blk = mode_block_index(a, ord_of(pf_tile));
        const int64_t rem = a.n_rows - blk * kTileM;
        pf_rows = rem < kTileM ? (int)rem : kTileM;
        pf_ptr = reinterpret_cast<const unsigned char*>(Eh + (size_t)(blk * kTileM + (lt & 127)) * a.ld);
        if (METRIC == RL_METRIC_COSINE && lt < 4 && lt * 32 < pf_rows) prefetch_l2(a.inv_norm + blk * kTileM + lt * 32);
      } else {
        pf_rows = 0;
      }
    };
    auto prefetch_item = [&]() {   // one 128-byte line per row and item
      if (lt < 128 && lt < pf_rows && pf_ks * kSliceK < a.d) prefetch_l2(pf_ptr);
      pf_ptr += slice_bytes;
      if (++pf_ks == t.n_ks) {
        pf_ks = 0;
        ++pf_tile;
        pf_set_tile();
      }
    };
    auto issue_item = [&](uint4 (&buf)[4]) {
      const bool col_ok = ld_ks * kSliceK + j * 8 < a.d;
      const unsigned char* p = ld_ptr;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (col_ok && r0 + 32 * i < ld_rows) buf[i] = ldg_stream_u4(p);
        else buf[i] = make_uint4(0u, 0u, 0u, 0u);
        p += pitch32_bytes;
      }
      ld_ptr += slice_bytes;
      if (++ld_ks == t.n_ks) {
        ld_ks = 0;
        ++ld_tile;
        ld_set_tile();
      }
      prefetch_item();
    };
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t sw_off = (uint32_t)r0 * 128u + (((uint32_t)j ^ ((uint32_t)r0 & 7u)) << 4);
    auto process = [&](uint4 (&buf)[4]) {
      mbar_wait(&s.empty[stage], phase ^ 1u);
      unsigned char* A = s.stage_base + (size_t)stage * sbytes + sw_off;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        *reinterpret_cast<uint4*>(A + i * 32 * 128) = buf[i];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.full[stage]);
      issue_item(buf);
      if (++stage == t.stages) { stage = 0; phase ^= 1u; }
    };
    ld_set_tile();
    pf_set_tile();
    for (int i = 0; i < 2 * kPrefetchItems; ++i) prefetch_item();
#pragma unroll
    for (int r = 0; r < 4; ++r) issue_item(ring[r]);
    for (int64_t item = 0; item < total_items; item += 4) {
      process(ring[0]);
      if (item + 1 < total_items) process(ring[1]);
      if (item + 2 < total_items) process(ring[2]);
      if (item + 3 < total_items) process(ring[3]);
    }
  } else if (warp >= kFirstLoaderWarp && fast_f32) {
    // ===== corpus loaders, fp32 storage, FAST PATH (d % 128 == 0, no per-row scale) =====
    // Same data movement as the generic loader below -- HBM fp32 -> registers (two K-slice items = 64 KB per SM in
    // flight) -> cvt.rn.f16x2 -> 128B-swizzled smem tile, L2 prefetch kPrefetchItems ahead -- with the bookkeeping
    // cut down.  ncu's source view of the generic loop showed ~155 SASS instructions per item and warp (three
    // cursors with 64-bit row pointers rebuilt per item, constants re-read from the parameter bank, the swizzle offset
    // rematerialised from %tid), and the loader warps, not memory, setting the pace at the power-capped SM clock:
    // 28 % "wait" + 15 % "selected" stall samples, a ~1000-cycle dependent chain per 1100-cycle item.  Here an
    // iteration handles the PAIR of items (ks, ks + 1): one cursor step, seven row pointers (32-bit pitch, one
    // IMAD.WIDE each) shared by both items through a +256 B immediate, smem / barrier addresses kept incrementally.
    const int lt = threadIdx.x - kFirstLoaderWarp * 32;  // 0..255
    const int c4 = lt & 15;                              // float4 column within the 64-wide K slice
    const int r0 = lt >> 4;                              // rows r0 + 16 i, i = 0..7
    const float gscale = (METRIC == RL_METRIC_COSINE) ? 1.f : pow2_scale(t.row_stats[1]);
    const bool mul = gscale != 1.f;
    uint32_t n_ks = (uint32_t)t.n_ks, n_stages = (uint32_t)t.stages;
    uint32_t pitch16 = (uint32_t)(a.ld * 16 * (int64_t)sizeof(float));   // bytes between this thread's consecutive rows
    uint32_t sw_off = (uint32_t)r0 * 128u + ((((uint32_t)c4 >> 1) ^ ((uint32_t)r0 & 7u)) << 4) + (((uint32_t)c4 & 1u) << 3);
    // opaque moves: keep these in registers instead of re-deriving them from %tid / the parameter bank per item
    asm volatile("" : "+r"(n_ks), "+r"(n_stages), "+r"(pitch16), "+r"(sw_off));
    const int64_t total_items = my_tiles * (int64_t)n_ks;

    struct Cursor { int64_t tile; uint32_t ks; int rows; const unsigned char* ptr; };
    // Load cursor: this thread's row r0 / column c4 of the NEXT pair of items to load.
    Cursor ld{0, 0u, 0, nullptr};
    auto ld_set_tile = [&]() {
      ld.rows = 0;
      if (ld.tile < my_tiles) {
        const int64_t ord = ord_of(ld.tile);
        if (ord < a.n_mode_blocks) {
          const int64_t blk = mode_block_index(a, ord);
          const int64_t rem = a.n_rows - blk * kTileM;
          ld.rows = rem < kTileM ? (int)rem : kTileM;
          ld.ptr = reinterpret_cast<const unsigned char*>(a.E + (size_t)(blk * kTileM + r0) * a.ld + c4 * 4);
        }
      }
    };
    // Prefetch cursor (L2 only): thread lt covers row lt / 2, 128-byte half lt % 2 of a 256-byte slice.
    Cursor pf{0, 0u, 0, nullptr};
    auto pf_set_tile = [&]() {
      pf.rows = 0;
      if (pg == 0 && pf.tile < my_tiles) {
        const int64_t ord = ord_of(pf.tile);
        if (ord < a.n_mode_blocks) {
          const int64_t blk = mode_block_index(a, ord);
          const int64_t rem = a.n_rows - blk * kTileM;
          pf.rows = rem < kTileM ? (int)rem : kTileM;
          pf.ptr = reinterpret_cast<const unsigned char*>(a.E + (size_t)(blk * kTileM + (lt >> 1)) * a.ld + (lt & 1) * 32);
          if (METRIC == RL_METRIC_COSINE && lt < 4 && lt * 32 < pf.rows) prefetch_l2(a.inv_norm + blk * kTileM + lt * 32);
        }
      }
    };
    auto pf_pair = [&]() {
      if ((lt >> 1) < pf.rows) { prefetch_l2(pf.ptr); prefetch_l2(pf.ptr + 256); }
      pf.ptr += 512;
      pf.ks += 2;
      if (pf.ks == n_ks) { pf.ks = 0; ++pf.tile; pf_set_tile(); }
    };
    float4 ringA[8], ringB[8];
    auto issue = [&](float4 (&buf)[8], int rows, const unsigned char* base) {   // base: row r0 of the item
      if (rows == kTileM) {   // full tile: no per-row predicates
#pragma unroll
        for (int i = 0; i < 8; ++i) buf[i] = ldg_stream(reinterpret_cast<const float*>(base + (size_t)((uint32_t)i * pitch16)));
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (r0 + 16 * i < rows) buf[i] = ldg_stream(reinterpret_cast<const float*>(base + (size_t)((uint32_t)i * pitch16)));
          else buf[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    // Store side: shared-memory addresses of the current stage, kept incrementally.
    uint32_t stage = 0, phase = 0;
    unsigned char* a_dst = s.stage_base + sw_off;
    auto store = [&](const float4 (&buf)[8]) {
      mbar_wait(&s.empty[stage], phase ^ 1u);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float4 v = buf[i];
        if (mul) { v.x *= gscale; v.y *= gscale; v.z *= gscale; v.w *= gscale; }
        const __half2 h01 = __floats2half2_rn(v.x, v.y);
        const __half2 h23 = __floats2half2_rn(v.z, v.w);
        uint2 packed;
        packed.x = *reinterpret_cast<const uint32_t*>(&h01);
        packed.y = *reinterpret_cast<const uint32_t*>(&h23);
        *reinterpret_cast<uint2*>(a_dst + i * 16 * 128) = packed;
      }
      // (no proxy fence here, see the generic loader: the MMA thread fences after acquiring the barrier)
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.full[stage]);
      a_dst += sbytes;
      if (++stage == n_stages) { stage = 0; phase ^= 1u; a_dst = s.stage_base + sw_off; }
    };

    ld_set_tile();
    pf_set_tile();
    for (int i = 0; i < kPrefetchPairs + 1; ++i) pf_pair();   // the load cursor starts one pair ahead of the stores
    issue(ringA, ld.rows, ld.ptr);
    issue(ringB, ld.rows, ld.ptr + 256);
    for (int64_t item = 0; item < total_items; item += 2) {
      // advance the load cursor to the next pair (possibly the first pair of the next tile)
      ld.ptr += 512;
      ld.ks += 2;
      if (ld.ks == n_ks) { ld.ks = 0; ++ld.tile; ld_set_tile(); }
      const int rows = ld.rows;
      const unsigned char* base = ld.ptr;
      store(ringA);
      issue(ringA, rows, base);
      store(ringB);
      issue(ringB, rows, base + 256);
      pf_pair();
    }
  } else if (warp >= kFirstLoaderWarp) {
    // ===== corpus loaders: HBM fp32 -> registers -> fp16 -> swizzled smem (UMMA A operand) =====
    const int lt = threadIdx.x - kFirstLoaderWarp * 32;  // 0..255
    const int c4 = lt & 15;                              // float4 column within the 64-wide K slice
    const int r0 = lt >> 4;                              // rows r0 + 16 i, i = 0..7
    const float gscale = (METRIC == RL_METRIC_COSINE) ? 1.f : pow2_scale(t.row_stats[1]);
    // Rows are converted without a multiply when no scaling is needed (normalised corpora: the
    // cosine 1/|e| then moves to the epilogue, which has slack; dot/l2: the global scale is 1).
    const bool noscale = (METRIC == RL_METRIC_COSINE) ? cos_noscale : (gscale == 1.f);
    const int64_t total_items = my_tiles * t.n_ks;
    float4 ring[2][8];
    float rs[8];

    // Incremental cursors (no integer divisions or multiplies on the hot path).  `ld_*` runs two items
    // ahead of `st_*`; `pf_*` runs kPrefetchItems ahead of `ld_*` and only touches L2.
    const size_t pitch16_bytes = (size_t)a.ld * 16 * sizeof(float);   // between this thread's consecutive rows
    const size_t slice_bytes = kSliceK * sizeof(float);
    int64_t ld_tile = 0;
    int ld_ks = 0, ld_rows = 0;
    const unsigned char* ld_ptr = nullptr;                 // row r0 of the tile, column c4*4 + ld_ks*64
    auto ld_set_tile = [&]() {
      if (ld_tile < my_tiles && ord_of(ld_tile) < a.n_mode_blocks) {
        const int64_t blk = mode_block_index(a, ord_of(ld_tile));
        const int64_t rem = a.n_rows - blk * kTileM;
        ld_rows = rem < kTileM ? (int)rem : kTileM;
        ld_ptr = reinterpret_cast<const unsigned char*>(a.E + (size_t)(blk * kTileM + r0) * a.ld + c4 * 4);
      } else {
        ld_rows = 0;
      }
    };
    // One 128-byte line per thread and item: thread lt covers row lt/2, half lt%2 of the 256-byte slice.
    int64_t pf_tile = 0;
    int pf_ks = 0, pf_rows = 0;
    const unsigned char* pf_ptr = nullptr;
    auto pf_set_tile = [&]() {   // only the first group's CTA of a lane prefetches
      if (pg == 0 && pf_tile < my_tiles && ord_of(pf_tile) < a.n_mode_blocks) {
        const int64_t blk = mode_block_index(a, ord_of(pf_tile));
        const int64_t rem = a.n_rows - blk * kTileM;
        pf_rows = rem < kTileM ? (int)rem : kTileM;
        pf_ptr = reinterpret_cast<const unsigned char*>(a.E + (size_t)(blk * kTileM + (lt >> 1)) * a.ld + (lt & 1) * 32);
        if (METRIC == RL_METRIC_COSINE && lt < 4 && lt * 32 < pf_rows) prefetch_l2(a.inv_norm + blk * kTileM + lt * 32);
      } else {
        pf_rows = 0;
      }
    };
    auto prefetch_item = [&]() {
      if ((lt >> 1) < pf_rows && pf_ks * kSliceK + (lt & 1) * 32 < a.d) prefetch_l2(pf_ptr);
      pf_ptr += slice_bytes;
      if (++pf_ks == t.n_ks) {
        pf_ks = 0;
        ++pf_tile;
        pf_set_tile();
      }
    };
    auto issue_item = [&](float4 (&buf)[8]) {
      const bool col_ok = ld_ks * kSliceK + c4 * 4 < a.d;
      const unsigned char* p = ld_ptr;
      if (col_ok && ld_rows == kTileM) {   // full tile: no per-row predicates
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          buf[i] = ldg_stream(reinterpret_cast<const float*>(p));
          p += pitch16_bytes;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          if (col_ok && r0 + 16 * i < ld_rows) buf[i] = ldg_stream(reinterpret_cast<const float*>(p));
          else buf[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          p += pitch16_bytes;
        }
      }
      ld_ptr += slice_bytes;
      if (++ld_ks == t.n_ks) {
        ld_ks = 0;
        ++ld_tile;
        ld_set_tile();
      }
      prefetch_item();
    };

    int64_t st_tile = 0;
    int st_ks = 0, stage = 0;
    uint32_t phase = 0;
    // Row scales of a tile are (re)loaded right after the last item of the previous tile has been
    // converted; their latency overlaps the arrive, the next loads and the next barrier wait.
    auto fetch_scales = [&](int64_t tile) {
#pragma unroll
      for (int i = 0; i < 8; ++i) rs[i] = (METRIC == RL_METRIC_COSINE) ? 0.f : gscale;
      if (METRIC == RL_METRIC_COSINE && !noscale && tile < my_tiles && ord_of(tile) < a.n_mode_blocks) {
        const int64_t blk = mode_block_index(a, ord_of(tile));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int64_t row = blk * kTileM + r0 + 16 * i;
          if (row < a.n_rows) rs[i] = __ldg(a.inv_norm + row);
        }
      }
    };
    // Per-thread constant part of the swizzled store offset: row r = r0 + 16 i has r & 7 == r0 & 7.
    const uint32_t sw_off = (uint32_t)r0 * 128u + ((((uint32_t)c4 >> 1) ^ ((uint32_t)r0 & 7u)) << 4) + (((uint32_t)c4 & 1u) << 3);
    // Convert + store one item, then refill its register slots with the loads of the item two
    // ahead: two stage-loads (64 KB per SM) stay in flight.
    auto process = [&](float4 (&buf)[8]) {
      mbar_wait(&s.empty[stage], phase ^ 1u);
      unsigned char* A = s.stage_base + (size_t)stage * sbytes + sw_off;
      if (noscale) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 h01 = __floats2half2_rn(buf[i].x, buf[i].y);
          const __half2 h23 = __floats2half2_rn(buf[i].z, buf[i].w);
          uint2 packed;
          packed.x = *reinterpret_cast<const uint32_t*>(&h01);
          packed.y = *reinterpret_cast<const uint32_t*>(&h23);
          *reinterpret_cast<uint2*>(A + i * 16 * 128) = packed;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 h01 = __floats2half2_rn(buf[i].x * rs[i], buf[i].y * rs[i]);
          const __half2 h23 = __floats2half2_rn(buf[i].z * rs[i], buf[i].w * rs[i]);
          uint2 packed;
          packed.x = *reinterpret_cast<const uint32_t*>(&h01);
          packed.y = *reinterpret_cast<const uint32_t*>(&h23);
          *reinterpret_cast<uint2*>(A + i * 16 * 128) = packed;
        }
      }
      // No proxy fence here: a fence in a thread with global loads in flight stalls until they land and
      // collapses the loaders' memory-level parallelism.  The stores are released by the mbarrier arrive;
      // the MMA thread acquires the barrier and executes fence.proxy.async before it issues tcgen05.mma.
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.full[stage]);
      issue_item(buf);
      if (++stage == t.stages) { stage = 0; phase ^= 1u; }
      if (++st_ks == t.n_ks) { st_ks = 0; ++st_tile; fetch_scales(st_tile); }
    };

    fetch_scales(0);
    ld_set_tile();
    pf_set_tile();
    for (int i = 0; i < kPrefetchItems; ++i) prefetch_item();
    issue_item(ring[0]);
    issue_item(ring[1]);
    for (int64_t item = 0; item < total_items; item += 2) {
      process(ring[0]);
      if (item + 1 < total_items) process(ring[1]);
    }
  } else if (warp == kQWarp) {
    // ===== query producer: bulk-copy the pre-swizzled fp16 K slice of all queries (UMMA B operand) =====
    if (lane == 0) {
      // The K slices of the group's nq queries follow each other in its image (nq * 128 bytes each).
      const uint32_t slice_bytes_q = (uint32_t)nq * 128u;
      const uint32_t qbytes = PAIR ? slice_bytes_q / 2 : slice_bytes_q;   // PAIR: this CTA's half of them
      const unsigned char* qsrc = reinterpret_cast<const unsigned char*>(qimg_g) + (PAIR ? (size_t)rank * qbytes : 0);
      const int64_t total_items = my_tiles * t.n_ks;
      int ks = 0, stage = 0;
      uint32_t phase = 0;
      // fp16 storage, tensor-map mode: this thread also brings the corpus tile -- row0 of the current tile (-1: this
      // CTA has no block for the tile, nothing is loaded and the epilogue ignores the accumulator) and of the
      // next one, whose slices are prefetched into L2 one tile (n_ks slices = 256 KB per SM at d = 1024) ahead.
      const bool tma_rows = EF16 && t.tma_rows;
      int64_t tile = 0;
      int row0 = -1, row0_next = -1;
      auto tile_row0 = [&](int64_t v) -> int {
        if (v >= my_tiles) return -1;
        const int64_t ord = ord_of(v);
        return ord < a.n_mode_blocks ? (int)(mode_block_index(a, ord) * kTileM) : -1;
      };
      if (tma_rows) { row0 = tile_row0(0); row0_next = tile_row0(1); }
      for (int64_t item = 0; item < total_items; ++item) {
        mbar_wait(&s.empty[stage], phase ^ 1u);
        const bool load_a = tma_rows && row0 >= 0;
        mbar_arrive_expect_tx(&s.full[stage], qbytes + (load_a ? (uint32_t)kABytes : 0u));
        if (load_a) tma_load_tile(s.stage_base + (size_t)stage * sbytes, &tmE, ks * kSliceK, row0, &s.full[stage]);
        bulk_g2s(s.stage_base + (size_t)stage * sbytes + kABytes, qsrc + (size_t)ks * slice_bytes_q, qbytes,
                 &s.full[stage]);
        if (tma_rows && row0_next >= 0 && pg == 0) tma_prefetch_tile(&tmE, ks * kSliceK, row0_next);
        if (++ks == t.n_ks) {
          ks = 0;
          if (tma_rows) { ++tile; row0 = row0_next; row0_next = tile_row0(tile + 1); }
        }
        if (++stage == t.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == kMmaWarp) {
    // ===== MMA issuer: one thread drives the tensor core =====
    if (PAIR && rank != 0) {
      // Peer CTA: no MMA issue.  Relay "my A tile and my half of the queries are in place" to the
      // leader's full barrier, stage by stage.
      if (lane == 0) {
        int stage = 0;
        uint32_t phase = 0;
        const int64_t total_items = my_tiles * t.n_ks;
        for (int64_t item = 0; item < total_items; ++item) {
          mbar_wait(&s.full[stage], phase);
          fence_proxy_async();
          mbar_arrive_remote(mapa_u32(&s.full[stage], 0));
          if (++stage == t.stages) { stage = 0; phase ^= 1u; }
        }
      }
    } else if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(PAIR ? 2 * kTileM : kTileM, nq);
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t tile = 0; tile < my_tiles; ++tile) {
        const int buf = (int)(tile & 1);
        if (PAIR) mbar_wait_cluster(&s.tmem_empty[buf], (uint32_t)(((tile >> 1) & 1) ^ 1));
        else mbar_wait(&s.tmem_empty[buf], (uint32_t)(((tile >> 1) & 1) ^ 1));
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * t.buf_cols);
        for (int ks = 0; ks < t.n_ks; ++ks) {
          if (PAIR) mbar_wait_cluster(&s.full[stage], phase);
          else mbar_wait(&s.full[stage], phase);
          fence_proxy_async();  // generic-proxy smem stores of the loaders -> async proxy (tensor core) reads
          tc_fence_after();
          const uint32_t a_addr = smem_u32(s.stage_base + (size_t)stage * sbytes);
          const uint64_t a_desc = make_kmajor_sw128_desc(a_addr);
          const uint64_t b_desc = make_kmajor_sw128_desc(a_addr + kABytes);
#pragma unroll
          for (int k = 0; k < kSliceK / 16; ++k) {
            // advance 16 fp16 = 32 bytes along K inside the swizzled row: +2 in the >>4 encoding
            if (PAIR) umma_f16_2cta(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (ks | k) != 0 ? 1u : 0u);
            else umma_f16(d_tmem, a_desc + (uint64_t)(2 * k), b_desc + (uint64_t)(2 * k), idesc, (ks | k) != 0 ? 1u : 0u);
          }
          // frees the smem stage (in both CTAs for PAIR) once these MMAs have read it
          if (PAIR) umma_commit_2cta(&s.empty[stage]);
          else umma_commit(&s.empty[stage]);
          if (++stage == t.stages) { stage = 0; phase ^= 1u; }
        }
        // accumulator complete -> epilogue (of both CTAs for PAIR)
        if (PAIR) umma_commit_2cta(&s.tmem_full[buf]);
        else umma_commit(&s.tmem_full[buf]);
      }
    }
  } else {
    // ===== epilogue warps 0..3: TMEM -> registers -> key -> dump / threshold + emit =====
    const int q = warp;  // TMEM lane quarter
    bool flushed_once = false;
    for (int64_t tile = 0; tile < my_tiles; ++tile) {
      const int buf = (int)(tile & 1);
      const int64_t ord = ord_of(tile);
      const bool has_block = ord < a.n_mode_blocks;
      const int64_t blk = has_block ? mode_block_index(a, ord) : 0;
      const int r_in = q * 32 + lane;
      const int64_t row = blk * kTileM + r_in;
      bool valid = has_block && row < a.n_rows;
      // rows the metadata filter masks out but that exist (not tombstoned): counted against the threshold when the
      // caller asks for the rank-then-filter bound (rl_maxsim_unfiltered_bound)
      bool masked_alive = false;
      if (valid && a.row_allowed != nullptr) {
        valid = a.row_allowed[row] != 0;
        if (!valid && a.cnt_all != nullptr) masked_alive = a.row_alive == nullptr || a.row_alive[row] != 0;
      }
      const float bias = (METRIC == RL_METRIC_L2 && valid) ? -a.sq_norm[row] : 0.f;
      const float lane_scale = (METRIC == RL_METRIC_COSINE && cos_noscale && valid) ? __ldg(a.inv_norm + row) : 1.f;
      mbar_wait(&s.tmem_full[buf], (uint32_t)((tile >> 1) & 1));
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * t.buf_cols);
      // Two register buffers: the TMEM load of chunk c+1 is in flight while chunk c is processed.
      auto process_chunk = [&](int c0, const uint32_t (&v)[32]) {
        if (a.dump_mode) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = c0 + j;
            if (col < a.B) {
              float key = __uint_as_float(v[j]);
              if (METRIC != RL_METRIC_COSINE) key = fmaf(key, s.cs[col], bias);
              else key *= lane_scale;
              if (has_block) a.dump[(size_t)col * a.n_sample_rows + ord * kTileM + r_in] = valid ? key : kNegInf;
            }
          }
        } else {
          // Two instructions per accumulator: the sign of  acc * scale - thr  (one FFMA; dot / l2: FFMA + FADD) is
          // shifted into a bit collector with one funnel shift -- element j ends up at bit 31 - j, set when the
          // key is BELOW its threshold (FMUL + FSETP + SEL took 3.5 per accumulator, DESIGN.md 3.1).  For cosine
          // the FFMA rounds once, so a key whose rounded product equals thr while the exact product lies below it
          // does not count as a hit; thr sits 2 eps (~1e-3) under anything the selection needs, a rounding step is 6e-8.
          uint32_t below = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float acc = __uint_as_float(v[j]);
            float tkey;
            if (METRIC != RL_METRIC_COSINE) tkey = fmaf(acc, s.cs[c0 + j], bias) - s.thr[c0 + j];
            else tkey = fmaf(acc, lane_scale, -s.thr[c0 + j]);
            below = __funnelshift_l(__float_as_uint(tkey), below, 1);
          }
          uint32_t mask = __brev(~below);   // bit j set <=> key j at or above its threshold
          if (masked_alive) {   // (only with RL_FLAG_COUNT_UNFILTERED on a filtered scan)
            uint32_t extra = mask;
            while (extra != 0) {
              const int j = __ffs(extra) - 1;
              extra &= extra - 1;
              atomicAdd(a.cnt_all + c0 + j, 1);
            }
          }
          if (!valid) mask = 0;
          while (mask != 0) {  // rare: a few hits per tile; picks v[j] with a register select tree
            const int j = __ffs(mask) - 1;
            mask &= mask - 1;
            const int col = c0 + j;
            float key = __uint_as_float(select32(v, j));
            if (METRIC != RL_METRIC_COSINE) key = fmaf(key, s.cs[col], bias);
            else key *= lane_scale;
            // Stage the hit in shared memory (one returning atomic for the slot; the histogram update
            // does not wait); per-query ranks and global slots are handed out in bulk at the flush.
            const int pos = atomicAdd(&s.list_n[0], 1);
            const int hb = col * kHistBins + hist_bin(key, s.thr0[col], s.inv_w[col]);
            atomicAdd(&s.hist[hb >> 1], 1u << ((hb & 1) * 16));
            if (pos < kListCap) {
              s.list[pos * 3 + 0] = (uint32_t)col;
              s.list[pos * 3 + 1] = __float_as_uint(key);
              s.list[pos * 3 + 2] = (uint32_t)row;
            } else {
              emit_candidate(a, col, key, (int32_t)row);
            }
          }
        }
      };
      uint32_t va[32], vb[32];
      tmem_ld32_async(taddr0, va);
      tmem_ld_wait(va);
      for (int c0 = 0; c0 < nq; c0 += 64) {
        const bool has_b = c0 + 32 < nq;
        if (has_b) tmem_ld32_async(taddr0 + (uint32_t)(c0 + 32), vb);
        process_chunk(c0, va);
        if (has_b) {
          tmem_ld_wait(vb);
          if (c0 + 64 < nq) tmem_ld32_async(taddr0 + (uint32_t)(c0 + 64), va);
          process_chunk(c0 + 32, vb);
          if (c0 + 64 < nq) tmem_ld_wait(va);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {  // TMEM buffer is free for tile + 2 (the leader CTA's barrier counts both epilogues)
        if (PAIR && rank != 0) mbar_arrive_remote(mapa_u32(&s.tmem_empty[buf], 0));
        else mbar_arrive(&s.tmem_empty[buf]);
      }
      if (!a.dump_mode) {
        // Staged hits are flushed when enough have accumulated (or after the last tile): one global
        // atomic per query that was hit since the previous flush, plus the staged histogram.  The two
        // barriers bracket the read of the counter so that all 128 epilogue threads decide alike.
        const int et = threadIdx.x;  // 0..127 (epilogue warps are warps 0..3)
        epi_bar_sync();
        const int n_all = s.list_n[0];
        epi_bar_sync();
        const bool last = tile + 1 == my_tiles;
        const bool do_flush = n_all >= (flushed_once ? kFlushAt : kFlushFirst) || (last && n_all > 0);
        if (do_flush) {
          flushed_once = true;
          const int n = min(n_all, kListCap);
          for (int e = et; e < n; e += kNumEpiWarps * 32) {   // rank of every staged hit within its query
            const int col = (int)s.list[e * 3 + 0];
            s.list[e * 3 + 0] = (uint32_t)col | ((uint32_t)atomicAdd(&s.cnt[col], 1) << 16);
          }
          epi_bar_sync();
          for (int col = et; col < kMaxQ; col += kNumEpiWarps * 32) {
            const int c = s.cnt[col];
            if (c > 0) {
              s.basev[col] = atomicAdd(a.cand_cnt + col, c);
              s.cnt[col] = 0;
            }
          }
          for (int w = et; w < kMaxQ * kHistBins / 2; w += kNumEpiWarps * 32) {
            const uint32_t h = s.hist[w];
            if (h != 0u) {
              if (h & 0xFFFFu) atomicAdd(a.ghist + 2 * w, (int)(h & 0xFFFFu));
              if (h >> 16) atomicAdd(a.ghist + 2 * w + 1, (int)(h >> 16));
              s.hist[w] = 0u;
            }
          }
          epi_bar_sync();
          if (et == 0) s.list_n[0] = 0;
          for (int e = et; e < n; e += kNumEpiWarps * 32) {
            const uint32_t w0 = s.list[e * 3 + 0];
            const int col = (int)(w0 & 0xFFFFu);
            const int slot = s.basev[col] + (int)(w0 >> 16);
            if (slot < a.cap)
              a.cand[(size_t)col * a.cap + slot] = Cand{__uint_as_float(s.list[e * 3 + 1]), (int32_t)s.list[e * 3 + 2]};
          }
        }
        const bool periodic = (tile % kRefreshEvery) == kRefreshEvery - 1;
        if ((do_flush || periodic) && !last) {
          // Threshold refresh: the highest bin edge with >= sel_count candidates at or above it (all
          // CTAs' hits so far) bounds the sel_count-th best key from below; emit from 2 eps under it.
          for (int col = et; col < a.B; col += kNumEpiWarps * 32) {
            const int4* gh = reinterpret_cast<const int4*>(a.ghist + (size_t)col * kHistBins);
            int cnts[kHistBins];
#pragma unroll
            for (int q4 = 0; q4 < kHistBins / 4; ++q4) {
              const int4 v4 = __ldcg(gh + q4);
              cnts[4 * q4] = v4.x; cnts[4 * q4 + 1] = v4.y; cnts[4 * q4 + 2] = v4.z; cnts[4 * q4 + 3] = v4.w;
            }
            int cum = 0, best = -1;
#pragma unroll
            for (int bb = kHistBins - 1; bb >= 1; --bb) {
              cum += cnts[bb];
              if (best < 0 && cum >= a.sel_count) best = bb;
            }
            if (best >= 1 && s.inv_w[col] > 0.f) {
              // edge = thr0 + best * w; new emission threshold = edge - 2 eps
              const float nt = s.thr0[col] + (float)best / s.inv_w[col] - 2.f * a.eps[col];
              if (nt > s.thr[col]) s.thr[col] = nt;
            }
          }
        }
        if (do_flush || periodic) epi_bar_sync();
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // the peer's smem / TMEM stay alive until the leader's last MMA has retired
  if (warp == kMmaWarp) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2cta(tmem_base, (uint32_t)t.tmem_cols);
    else tmem_dealloc(tmem_base, (uint32_t)t.tmem_cols);
  }
}

// Query image: fp16, scaled, laid out exactly as the swizzled smem stage rows.
__global__ void __launch_bounds__(128) query_image_kernel(const float* __restrict__ Q, int B, int d, int metric,
                                                          const float* __restrict__ q_inv_norm,
                                                          const float* __restrict__ row_stats, float* __restrict__ q_scale,
                                                          __half* __restrict__ qimg, int n_ks, int rows_scaled) {
  __shared__ float red[4];
  const int b = blockIdx.x;
  const int group = b / kMaxQ, n = b % kMaxQ;
  const int nq = min(kMaxQ, (B - group * kMaxQ + 15) / 16 * 16);
  const float* q = Q + (size_t)b * d;
  float scale;
  if (metric == RL_METRIC_COSINE) {
    scale = q_inv_norm[b];
    if (threadIdx.x == 0) q_scale[b] = 1.f;
  } else {
    float m = 0.f;
    for (int c = threadIdx.x; c < d; c += blockDim.x) m = fmaxf(m, fabsf(q[c]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    scale = pow2_scale(m);
    // the loaders of an fp32 corpus multiply the rows by a global power of two (dot / l2); fp16-stored rows stay as they are
    const float rs_e = rows_scaled ? pow2_scale(row_stats[1]) : 1.f;
    if (threadIdx.x == 0) q_scale[b] = (metric == RL_METRIC_L2 ? 2.f : 1.f) / (scale * rs_e);
  }
  __half* img = qimg + (size_t)group * n_ks * kMaxQ * kSliceK;  // groups are laid out with the full 256-row pitch
  for (int c = threadIdx.x; c < n_ks * kSliceK; c += blockDim.x) {
    const int ks = c / kSliceK, e = c % kSliceK;
    const float v = c < d ? q[c] * scale : 0.f;
    const int chunk = e >> 3, within = e & 7;
    const size_t off = ((size_t)ks * nq + n) * kSliceK + (size_t)(((chunk ^ (n & 7)) << 3) + within);
    img[off] = __float2half_rn(v);
  }
}

}  // namespace

bool tcgen05_supported(const rl_scan_params* p) {
  if (p == nullptr || p->n_rows <= 0 || p->B <= 0) return false;
  if (p->e_dtype == 1 && (p->d % 8 != 0 || p->ld % 8 != 0)) return false;
  if (p->d % 4 != 0 || p->ld % 4 != 0) return false;
  if ((reinterpret_cast<uintptr_t>(p->E) & 15) != 0) return false;
  if ((p->d + kSliceK - 1) / kSliceK > 1024) return false;
  return true;
}

size_t tcgen05_qimg_bytes(int B, int d) {
  const int n_ks = (d + kSliceK - 1) / kSliceK;
  const int groups = (B + kMaxQ - 1) / kMaxQ;
  return (size_t)groups * n_ks * kMaxQ * kSliceK * sizeof(__half);
}

int tcgen05_prepare_queries(const rl_scan_params* p, const float* q_inv_norm, float* q_scale, void* qimg,
                            cudaStream_t stream) {
  const int n_ks = (p->d + kSliceK - 1) / kSliceK;
  RL_CUDA_CHECK(cudaMemsetAsync(qimg, 0, tcgen05_qimg_bytes(p->B, p->d), stream));
  query_image_kernel<<<p->B, 128, 0, stream>>>(p->Q, p->B, p->d, p->metric, q_inv_norm, p->row_stats, q_scale,
                                                 reinterpret_cast<__half*>(qimg), n_ks, p->e_dtype == 1 ? 0 : 1);
  RL_CUDA_CHECK(cudaGetLastError());
  return RL_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency).
typedef CUresult (*ScanEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                      const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static ScanEncodeTiledFn scan_encode_tiled_fn() {
  static ScanEncodeTiledFn fn = []() -> ScanEncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<ScanEncodeTiledFn>(p);
  }();
  return fn;
}
// Tensor map over the fp16-stored corpus E[n_rows, ld] (d valid columns): box = 64 halves (one 128-byte swizzle row)
// x 128 rows = exactly one UMMA A stage; rows past n_rows and columns past d read as zero.
static bool make_corpus_tensor_map(CUtensorMap* tm, const void* E, int64_t n_rows, int64_t ld, int d) {
  ScanEncodeTiledFn enc = scan_encode_tiled_fn();
  if (enc == nullptr || (reinterpret_cast<uintptr_t>(E) & 15) != 0 || (ld * 2) % 16 != 0 || n_rows >= (int64_t(1) << 31)) return false;
  const cuuint64_t gdim[2] = {(cuuint64_t)d, (cuuint64_t)n_rows};
  const cuuint64_t gstr[1] = {(cuuint64_t)ld * sizeof(__half)};
  const cuuint32_t box[2] = {(cuuint32_t)kSliceK, (cuuint32_t)kTileM};
  const cuuint32_t estr[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(E), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr int kMaxGroups = 4;   // query groups per launch (B <= 1024 per launch)

int launch_scan_tcgen05(const ScanArgs& a_in, const rl_scan_params* p, const float* q_scale, const void* qimg,
                        int sm_count, cudaStream_t stream) {
  if (a_in.n_mode_blocks == 0 || a_in.B == 0) return RL_OK;
  const int n_ks = (p->d + kSliceK - 1) / kSliceK;
  const int groups = (a_in.B + kMaxQ - 1) / kMaxQ;
  // The groups of 256 queries of one launch run group-parallel: the CTAs of a lane walk the same tiles at the
  // same time, one group each, and meet in L2, so HBM sees the corpus once (configs[2], B = 1024).  A lane needs
  // at least two SMs per group, which caps the groups per launch.
  const int max_groups = min(kMaxGroups, max(1, sm_count / 2));
  // fp16 storage: the corpus tiles go HBM -> shared memory through a tensor map (TMA writes the swizzled UMMA tile,
  // no loader warps, no registers in between); the register loaders take the corpora a tensor map cannot describe.
  CUtensorMap tmE;
  memset(&tmE, 0, sizeof(tmE));
  const bool tma_rows = p->e_dtype == 1 && make_corpus_tensor_map(&tmE, p->E, p->n_rows, p->ld, p->d);
  for (int g0 = 0; g0 < groups; g0 += max_groups) {
    TcArgs t;
    t.a = a_in;
    const int q0 = g0 * kMaxQ;
    const int ng = groups - g0 < max_groups ? groups - g0 : max_groups;
    const int nb = a_in.B - q0 < ng * kMaxQ ? a_in.B - q0 : ng * kMaxQ;
    t.a.B = nb;
    t.a.thr = a_in.thr + q0;
    t.a.dump = a_in.dump + (size_t)q0 * a_in.n_sample_rows;
    t.a.cand = a_in.cand + (size_t)q0 * a_in.cap;
    t.a.cand_cnt = a_in.cand_cnt + q0;
    t.a.ghist = a_in.ghist + (size_t)q0 * kHistBins;
    t.a.eps = a_in.eps + q0;
    t.a.hist_inv_w = a_in.hist_inv_w + q0;
    t.a.q_inv_norm = a_in.q_inv_norm + q0;
    t.a.cnt_all = a_in.cnt_all ? a_in.cnt_all + q0 : nullptr;
    t.qimg = reinterpret_cast<const __half*>(qimg) + (size_t)g0 * n_ks * kMaxQ * kSliceK;
    t.q_scale = q_scale + q0;
    t.row_stats = p->row_stats;
    t.par_groups = ng;
    const int last_b = nb - (ng - 1) * kMaxQ;              // queries of the last group
    t.nq_last = (last_b + 15) / 16 * 16;
    t.nq = ng > 1 ? kMaxQ : t.nq_last;                     // a full group (the only group when ng == 1)
    t.n_ks = n_ks;
    t.tma_rows = tma_rows ? 1 : 0;
    t.buf_cols = (t.nq + 31) / 32 * 32;
    int cols = 32;
    while (cols < 2 * t.buf_cols) cols *= 2;
    t.tmem_cols = cols;
    // cta_group::2 (SM pair): the two CTAs of a cluster issue ONE M = 256 MMA per K step and each holds only half
    // of the query slice, so an SM pulls 16 KB instead of 32 KB of query image per stage from L2 (the L2 -> SM
    // stream: -25 % on an fp32 corpus, -33 % on fp16).  Used for a single query group (B <= 256); the barrier
    // operations in its hot loop are default-scope, since the cluster-scope ones compile to MEMBAR.ALL.GPU /
    // CCTL.IVALL.  Group-parallel lanes (B > 256) do not gain from pairs and keep one CTA per SM (DESIGN.md 3.1).
    const bool pair = ng == 1 && t.nq % 32 == 0 && t.nq_last % 32 == 0 && t.nq_last >= 64 && a_in.n_mode_blocks >= 2 &&
                      sm_count >= 2;
    const uint32_t avail = kSmemBudget - 1024 - tail_bytes();
    int stages = (int)(avail / stage_bytes(pair ? t.nq / 2 : t.nq));
    if (stages > kMaxStages) stages = kMaxStages;
    RL_REQUIRE(stages >= 2, RL_EUNSUPPORTED, "tcgen05 scan: not enough shared memory for 2 stages");
    t.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes(pair ? t.nq / 2 : t.nq) + tail_bytes() + 1024;
    RL_REQUIRE(p->row_stats != nullptr, RL_EINVAL, "tcgen05 scan needs row_stats");
    auto launch = [&](auto kernel, bool is_pair) -> int {
      RL_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      cudaLaunchConfig_t cfg{};
      cudaLaunchAttribute attr[1];
      if (is_pair) {
        const int64_t n_pairs = (a_in.n_mode_blocks + 1) / 2;
        const int units = sm_count / 2 / t.par_groups;                  // lanes of par_groups clusters each
        const int clusters = (int)(n_pairs < units ? n_pairs : units) * t.par_groups;
        cfg.gridDim = dim3((unsigned)(2 * clusters));
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
      } else {
        const int lanes = sm_count / t.par_groups;
        cfg.gridDim = dim3((unsigned)((a_in.n_mode_blocks < lanes ? a_in.n_mode_blocks : lanes) * t.par_groups));
      }
      cfg.blockDim = dim3(kThreads);
      cfg.dynamicSmemBytes = smem;
      cfg.stream = stream;
      RL_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, tmE, t));
      return RL_OK;
    };
    int rc;
    const bool f16 = p->e_dtype == 1;
    auto dispatch = [&](auto metric_tag) -> int {
      constexpr int M = decltype(metric_tag)::value;
      if (pair) return f16 ? launch(scan_tcgen05_kernel<M, true, true>, true) : launch(scan_tcgen05_kernel<M, true, false>, true);
      return f16 ? launch(scan_tcgen05_kernel<M, false, true>, false) : launch(scan_tcgen05_kernel<M, false, false>, false);
    };
    if (p->metric == RL_METRIC_COSINE) rc = dispatch(std::integral_constant<int, RL_METRIC_COSINE>{});
    else if (p->metric == RL_METRIC_DOT) rc = dispatch(std::integral_constant<int, RL_METRIC_DOT>{});
    else rc = dispatch(std::integral_constant<int, RL_METRIC_L2>{});
    if (rc != RL_OK) return rc;
  }
  return RL_OK;
}

}  // namespace rl
