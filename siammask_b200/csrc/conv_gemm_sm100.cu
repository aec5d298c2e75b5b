// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05) for sm_100a.
//
//   out[m][n] = epilogue( sum_k A[m][k] * W[n][k] ),  m = (b, ho, wo) flattened, k = (r, s, c) with c fastest.
//
// * A (NHWC fp16 activation planes) is staged by TMA: plain 2-D tiles for 1x1/stride-1 convs, im2col-mode
//   tiles (cp.async.bulk.tensor.4d...im2col) for everything else — padding, stride and dilation are resolved
//   by the TMA unit, out-of-image taps arrive as zeros, and the 128-pixel M tile runs across row and image
//   boundaries so batch absorbs the odd spatial sizes (31x31, 29x29, 25x25 ...).
// * W (K-major fp16, [Cout_pad][KH*KW*Cin]) is staged by 2-D TMA tiles.  Both land in 128B-swizzled smem
//   and are consumed by tcgen05.mma (M=128, N=BLOCK_N, K=16) issued by a single thread; accumulators live
//   in TMEM, double-buffered so the epilogue of tile i overlaps the main loop of tile i+1.
// * Precision: NSPLIT=1 multiplies the fp16 hi planes only.  NSPLIT=2 ("exact") keeps activations and
//   weights as hi+lo fp16 pairs (22 significant bits) and issues three MMAs per k-step
//   (hi*hi into one TMEM accumulator, lo*hi + hi*lo into a second one, summed in the epilogue) — fp32-class
//   results from the fp16 tensor pipe.
// * Epilogue (8 warps, two per TMEM lane quarter, alternating 32-column chunks): tcgen05.ld -> acc*alpha[c]+beta[c]
//   (ReLU) -> NHWC split-fp16 planes through 64B-swizzled smem and TMA stores (direct stores would touch 32
//   sectors per request), or NHWC fp32, or NCHW fp32 (the boundary layout of the reference's outputs,
//   tools/test.py:205-206) — TMEM lanes are pixels, so NCHW stores are coalesced across the warp.
//
// * K may consist of up to two SEGMENTS that accumulate into the same tile: (conv over input 0) + (conv over
//   input 1) fuses a bottleneck's downsample branch with its conv3, and an IDENTITY segment
//   acc += residual * diag(2^e) streams the residual tensor through the same TMA/MMA pipeline (one extra
//   k-block per 64 output columns) instead of stalling the epilogue on it.
//
// Warp roles (320 threads): warp 0 = TMA producer (one lane), warp 1 = TMEM owner + MMA issuer (one lane),
// warps 2..9 = epilogue (two per TMEM lane quarter).  Persistent: grid = min(tiles, SMs), static round-robin over (m_tile, n_tile).
//
// * CG = 2 runs the same kernel as a CTA PAIR (cluster of two, tcgen05 cta_group::2) on a 256 x BLOCK_N tile: each CTA
//   stages its own 128 A rows and half of the B rows (TMA loads of both CTAs signal the leader's full barrier), the
//   leader's MMA thread issues M=256 instructions that write both CTAs' TMEM and multicasts its commits to the pair's
//   empty / accumulator-full barriers, the epilogue warps of both CTAs release the accumulator on the leader's barrier.
//   Per flop this moves a third less through each SM's shared-memory port, the resource that caps the single-CTA
//   exact-mode tiles at ~65 % tensor duty (see launch_gemm_multi for the tile choice and the measurements).
#include "common.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <cstring>
#include <mutex>
#include <unordered_map>

namespace smk {

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;     // k-block width in fp16 elements: one 128-byte swizzled row
constexpr int CIN_GRAIN = 64;  // convs need Cin % 64 == 0 (whole k-blocks per filter tap)
constexpr int UMMA_K = 16;
constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int NUM_EPI_WARPS = 8;   // two per TMEM lane quarter, alternating 32-column chunks
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;

// CG = CTAs per tile: 1, or 2 = a CTA pair (cluster of 2, tcgen05 cta_group::2) computing a 256 x BLOCK_N tile — each
// CTA stages its own 128 A rows and HALF of the B rows, so smem fill and MMA operand reads per flop drop by a third.
template <int BLOCK_N, int NSPLIT, int CG = 1>
struct Cfg {
  static constexpr int A_TILE_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_ROWS = BLOCK_N / CG;           // B rows staged by one CTA
  static constexpr int B_TILE_BYTES = B_ROWS * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = NSPLIT * (A_TILE_BYTES + B_TILE_BYTES);
  // epilogue staging: 8 warps x NSPLIT planes x (32 rows x 64 B)
  static constexpr int STG_TILE_BYTES = 32 * 64;
  static constexpr int STG_WARP_BYTES = NSPLIT * STG_TILE_BYTES;
  static constexpr int STG_BYTES = BLOCK_N >= 32 ? NUM_EPI_WARPS * STG_WARP_BYTES : 0;
  static constexpr int RAW_STAGES = (SMEM_LIMIT - 2048 - STG_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 6 ? 6 : RAW_STAGES;
  // 2 pipeline stages x NSPLIT accumulators (exact mode keeps the hi*hi sum and the 2^-11-sized cross terms in
  // separate TMEM accumulators: the tensor pipe truncates on every accumulate, so feeding small terms into the
  // large running sum — or tripling the number of adds into it — costs accuracy; they are summed in the epilogue)
  static constexpr int ACC_COLS = NSPLIT * BLOCK_N;
  // two accumulator stages (epilogue of tile i overlaps the main loop of tile i+1) when TMEM allows, else one
  static constexpr int ACC_STAGES = 2 * ACC_COLS <= 512 ? 2 : 1;
  static constexpr int ACC_TOTAL = ACC_STAGES * ACC_COLS;
  static constexpr int TMEM_COLS = (ACC_TOTAL <= 32) ? 32 : (ACC_TOTAL <= 64) ? 64 : (ACC_TOTAL <= 128) ? 128
                                   : (ACC_TOTAL <= 256) ? 256 : 512;
  static_assert(ACC_TOTAL <= 512, "TMEM capacity");
  static constexpr int CH = BLOCK_N < 32 ? 16 : 32;   // epilogue column chunk
  // one CTA per SM: keep the request above half of the SM's shared memory
  static constexpr int SMEM_BYTES_RAW = STAGES * STAGE_BYTES + STG_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
  static constexpr int SMEM_BYTES = SMEM_BYTES_RAW < 120 * 1024 ? 120 * 1024 : SMEM_BYTES_RAW;
  static_assert(STAGES >= 2, "pipeline needs at least two stages");
  static_assert(BLOCK_N % 16 == 0 && BLOCK_N >= 16 && BLOCK_N <= 256, "UMMA N constraint for M=128");
  static_assert(CG == 1 || (CG == 2 && BLOCK_N >= 64 && B_ROWS % 8 == 0), "CTA pairs: N >= 64");
  static_assert(SMEM_BYTES <= SMEM_LIMIT, "shared memory budget");
};

template <int CH>
__device__ __forceinline__ void tmem_ld_chunk(uint32_t taddr, uint32_t (&r)[CH]) {
  if constexpr (CH == 32) tmem_ld_32x32b_x32(taddr, r);
  else tmem_ld_32x32b_x16(taddr, r);
}

// tile -> M block.  With reverse_m the persistent CTAs walk the M tiles from the end: a layer then starts on the rows
// its producer wrote last, which are the ones still resident in the 126 MB L2 (activations of 250 MB stream through).
// With CTA pairs a tile covers CG consecutive M blocks; `rank` picks this CTA's.  The result may be == m_tiles for
// the odd last block of a pair (the caller clamps its loads and skips its stores).
template <int CG>
__device__ __forceinline__ int m_block(const GemmParams& p, int tile, int rank) {
  const int groups = (p.m_tiles + CG - 1) / CG;
  const int mb = tile / p.n_tiles;
  return (p.reverse_m ? groups - 1 - mb : mb) * CG + rank;
}

template <int BLOCK_N, int NSPLIT, int CG>
__global__ void __launch_bounds__(NUM_THREADS, 1) conv_gemm_kernel(const __grid_constant__ GemmParams p) {
  using C = Cfg<BLOCK_N, NSPLIT, CG>;
  constexpr int STAGES = C::STAGES;
  constexpr int CH = C::CH;
  constexpr int A_TILE_BYTES = C::A_TILE_BYTES;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stg_base = smem + STAGES * C::STAGE_BYTES;                      // 1024-aligned (stage sizes are)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stg_base + C::STG_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  // warp index through a shuffle: provably warp-uniform for the compiler, so the role branches below are convergent.
  // Every role loop is walked by its WHOLE warp and a single elected lane issues the TMA / tcgen05 instructions: their
  // operands live in uniform registers, and under a `threadIdx.x == k` branch ptxas wraps each of them in a
  // divergence loop (ELECT / R2UR / BRA per instruction — ~90 clk of issue time per MMA: slower than the 32..64 tensor
  // clocks of an N = 64..128 MMA).
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const bool leader = elect_one();
  const int rank = CG == 2 ? static_cast<int>(cluster_ctarank()) : 0;   // position in the CTA pair; 0 = leader
  const int num_tiles = ((p.m_tiles + CG - 1) / CG) * p.n_tiles;
  const int tile0 = blockIdx.x / CG;
  const int tile_step = gridDim.x / CG;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSPLIT; ++i) {
      for (int sgi = 0; sgi < p.nseg; ++sgi) tma_prefetch_desc(&p.seg[sgi].tmA[i]);
      tma_prefetch_desc(&p.tmB[i]);
    }
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], CG * NUM_EPI_WARPS);   // one arrival per epilogue warp (of both CTAs of a pair)
    }
    if (p.staged)
      for (int i = 0; i < NSPLIT; ++i) tma_prefetch_desc(&p.tmOut[i]);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) {
    __syncwarp();
    if constexpr (CG == 2) tmem_alloc_pair<C::TMEM_COLS>(tmem_slot);
    else tmem_alloc<C::TMEM_COLS>(tmem_slot);
  }
  tcgen05_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();      // the peer's barriers are initialised before anything signals them
  tcgen05_fence_after();
  // broadcast through a shuffle so the compiler KNOWS the TMEM base is warp-uniform: tcgen05 operands live in uniform
  // registers, and a value that merely came out of shared memory makes ptxas wrap every single MMA in a
  // divergence ("waterfall") loop — ELECT / R2UR / branch per instruction, ~90 clk of issue time per MMA
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  if (warp == 0) {
    // ===================== TMA producer =====================
    // CTA pairs: both producers fill their own smem but signal the LEADER's full barrier, which expects the bytes of
    // both CTAs; each waits on its own empty barrier (the leader's tcgen05.commit is multicast to the pair).
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t full0 = CG == 2 ? mapa_shared(smem_u32(&full_bar[0]), 0) : 0;
    auto acquire = [&](uint32_t bytes_per_cta) {
      if constexpr (CG == 2) mbar_wait_guarded(&empty_bar[stage], phase ^ 1);
      else mbar_wait(&empty_bar[stage], phase ^ 1);
      if (rank == 0 && leader) mbar_arrive_expect_tx(&full_bar[stage], CG * bytes_per_cta);
    };
    auto load_2d = [&](void* dst, const CUtensorMap* map, int c0, int c1) {
      if (!leader) return;
      if constexpr (CG == 2) tma_load_2d_pair(dst, map, full0 + stage * 8, c0, c1);
      else tma_load_2d(dst, map, &full_bar[stage], c0, c1);
    };
    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
      const int mb = m_block<CG>(p, tile, rank);
      const int m0 = (mb < p.m_tiles ? mb : p.m_tiles - 1) * BLOCK_M;   // odd last block of a pair: reload, never stored
      const int n0 = (tile % p.n_tiles) * BLOCK_N;
      const int nb0 = n0 + rank * C::B_ROWS;                            // first B row this CTA stages
      const int q = m0 % p.Wo;
      const int t = m0 / p.Wo;
      const int pq = t % p.Ho;
      const int nb = t / p.Ho;
      for (int sgi = 0; sgi < p.nseg; ++sgi) {
        const GemmSegment& sg = p.seg[sgi];
        if (sg.kind == 1) {
          // identity segment: A = residual tile [128 rows x 64 cols] (K-major), B = diag(2^e) block (hi plane only)
#pragma unroll 1
          for (int kb = 0; kb < BLOCK_N / BLOCK_K; ++kb) {
            acquire(NSPLIT * A_TILE_BYTES + C::B_TILE_BYTES);
            uint8_t* st = smem + stage * C::STAGE_BYTES;
#pragma unroll
            for (int s = 0; s < NSPLIT; ++s) load_2d(st + s * A_TILE_BYTES, &sg.tmA[s], n0 + kb * BLOCK_K, m0);
            load_2d(st + NSPLIT * A_TILE_BYTES, &p.tmB[0], sg.b_col0 + n0 + kb * BLOCK_K, nb0);
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          continue;
        }
        const int wb = q * sg.stride - sg.pad;
        const int hb = pq * sg.stride - sg.pad;
#pragma unroll 1
        for (int kb = 0; kb < sg.num_kb; ++kb) {
          acquire(C::STAGE_BYTES);
          uint8_t* st = smem + stage * C::STAGE_BYTES;
          const int tap = kb / sg.cblks;
          const int c0 = (kb - tap * sg.cblks) * BLOCK_K;
#pragma unroll
          for (int s = 0; s < NSPLIT; ++s) {
            uint8_t* a_dst = st + s * A_TILE_BYTES;
            if (sg.mode == 0) {
              load_2d(a_dst, &sg.tmA[s], c0, m0);
            } else {
              const int r = tap / sg.KW;
              const int sx = tap - r * sg.KW;
              if (leader) {
                if constexpr (CG == 2)
                  tma_load_im2col_4d_pair(a_dst, &sg.tmA[s], full0 + stage * 8, c0, wb, hb, nb,
                                          static_cast<uint16_t>(sx * sg.dil), static_cast<uint16_t>(r * sg.dil));
                else
                  tma_load_im2col_4d(a_dst, &sg.tmA[s], &full_bar[stage], c0, wb, hb, nb,
                                     static_cast<uint16_t>(sx * sg.dil), static_cast<uint16_t>(r * sg.dil));
              }
            }
            uint8_t* b_dst = st + NSPLIT * A_TILE_BYTES + s * C::B_TILE_BYTES;
            load_2d(b_dst, &p.tmB[s], sg.b_col0 + kb * BLOCK_K, nb0);
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    if constexpr (CG == 2) {
      // tail: every multicast commit aimed at this CTA's empty barriers has landed before it may exit
      for (int i = 0; i < STAGES; ++i) {
        mbar_wait_guarded(&empty_bar[stage], phase ^ 1);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===================== MMA issuer (pairs: the leader CTA issues for both) =====================
    constexpr uint32_t idesc = umma_idesc_f16(BLOCK_M * CG, BLOCK_N);
    // exact single-CTA tiles issue hi*hi and hi*lo as one MMA over [B_hi; B_lo] (see below); the pair tile keeps
    // three MMAs per k-step, since its N = 256 leaves no room for the concatenated operand
    constexpr bool NCAT = NSPLIT == 2 && CG == 1;
    static_assert(!NCAT || 2 * BLOCK_N <= 256, "concatenated MMA: N <= 256");
    constexpr uint32_t idesc_cat = umma_idesc_f16(BLOCK_M, NCAT ? 2 * BLOCK_N : BLOCK_N);
    auto wait_bar = [&](uint64_t* bar, uint32_t parity) {
      if constexpr (CG == 2) mbar_wait_guarded(bar, parity);
      else mbar_wait(bar, parity);
    };
    auto mma = [&](uint32_t d, uint64_t da, uint64_t db, uint32_t accumulate) {
      if constexpr (CG == 2) umma_f16_pair(d, da, db, idesc, accumulate);
      else umma_f16(d, da, db, idesc, accumulate);
    };
    auto commit = [&](uint64_t* bar) {
      if constexpr (CG == 2) umma_commit_pair(bar);
      else umma_commit(bar);
    };
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int tile = tile0; tile < num_tiles; tile += tile_step, ++it) {
      const int acc = it % C::ACC_STAGES;
      const uint32_t acc_phase = (it / C::ACC_STAGES) & 1;
      wait_bar(&tempty_bar[acc], acc_phase ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + acc * C::ACC_COLS;
      uint32_t acc_main = 0, acc_lo = 0;     // 0 on the first MMA into each accumulator of this tile
      for (int sgi = 0; sgi < p.nseg; ++sgi) {
        const GemmSegment& sg = p.seg[sgi];
        const bool ident = sg.kind == 1;
        const int nkb = ident ? BLOCK_N / BLOCK_K : sg.num_kb;
        const bool last_seg = sgi == p.nseg - 1;
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb) {
          wait_bar(&full_bar[stage], phase);
          tcgen05_fence_after();
          const uint32_t a_hi = smem_u32(smem + stage * C::STAGE_BYTES);
          const uint32_t b_hi = a_hi + NSPLIT * A_TILE_BYTES;
          // descriptors once per k-block; the K steps add (16 elements * 2 B) >> 4 = 2 to the start-address field
          const uint64_t da_hi0 = umma_desc_kmajor_sw128(a_hi);
          const uint64_t db_hi0 = umma_desc_kmajor_sw128(b_hi);
          const uint64_t da_lo0 = umma_desc_kmajor_sw128(a_hi + A_TILE_BYTES);
          const uint64_t db_lo0 = umma_desc_kmajor_sw128(b_hi + C::B_TILE_BYTES);
          if (leader) {
            if (NCAT && !ident) {
              // The B_lo tile follows the B_hi tile in the stage, so [B_hi; B_lo] is one K-major operand of 2*BLOCK_N
              // rows and the two accumulators are adjacent TMEM columns: A_hi x [B_hi; B_lo] is ONE MMA (hi*hi ->
              // acc0, hi*lo -> acc1) and A_hi crosses the shared-memory port once instead of twice (operand reads
              // per k-block 96 -> 80 KB at 128 x 128).  Both accumulate flags are always equal (set together).
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                const uint64_t kadd = static_cast<uint64_t>(k * UMMA_K * 2 / 16);
                umma_f16(tmem_d, da_hi0 + kadd, db_hi0 + kadd, idesc_cat, acc_main);
                acc_main = 1;
                mma(tmem_d + BLOCK_N, da_lo0 + kadd, db_hi0 + kadd, 1u);
              }
            } else {
#pragma unroll
              for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
                const uint64_t kadd = static_cast<uint64_t>(k * UMMA_K * 2 / 16);
                mma(tmem_d, da_hi0 + kadd, db_hi0 + kadd, acc_main);
                acc_main = 1;
                if constexpr (NSPLIT == 2) {
                  // same order as the concatenated form (hi*lo, then lo*hi): every tile variant rounds identically
                  if (!ident) {
                    mma(tmem_d + BLOCK_N, da_hi0 + kadd, db_lo0 + kadd, acc_lo);
                    acc_lo = 1;
                  }
                  mma(tmem_d + BLOCK_N, da_lo0 + kadd, db_hi0 + kadd, acc_lo);
                  acc_lo = 1;
                }
              }
            }
            commit(&empty_bar[stage]);                                   // smem slot free once these MMAs retire
            if (last_seg && kb == nkb - 1) commit(&tfull_bar[acc]);      // accumulator complete
          }
          __syncwarp();
          acc_main = 1;
          acc_lo = 1;
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 2) {
    // ===================== epilogue =====================
    const int quarter = warp & 3;             // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;         // which of the quarter's two warps: takes every other chunk
    const Epilogue& ep = p.ep;
    const int HoWo = p.Ho * p.Wo;
    int it = 0;
    // pairs: the accumulator stage is released to the LEADER's MMA thread by the epilogue warps of both CTAs
    const uint32_t tempty0 = CG == 2 ? mapa_shared(smem_u32(&tempty_bar[0]), 0) : 0;
    auto wait_acc = [&](uint64_t* bar, uint32_t parity) {
      if constexpr (CG == 2) mbar_wait_guarded(bar, parity);
      else mbar_wait(bar, parity);
    };
    auto release_acc = [&](int acc) {
      if constexpr (CG == 2) mbar_arrive_cluster(tempty0 + acc * 8);
      else mbar_arrive(&tempty_bar[acc]);
    };
    if constexpr (BLOCK_N >= 32) {
      if (p.staged) {
        // ---- staged path: TMEM -> registers -> 64B-swizzled smem -> TMA store.  Two warps share each block of 32
        // output rows and alternate 32-column chunks, each with its own staging buffer, so one warp's store and
        // TMEM latency overlap the other's math.  (A residual, if any, was accumulated by the identity segment.)
        uint8_t* buf = stg_base + (warp - 2) * C::STG_WARP_BYTES;
        constexpr int CHUNKS = BLOCK_N / 32;
        const int swz = (lane >> 1) & 3;                       // Swizzle<2,4,3>: 16B chunk ^= (row >> 1) & 3
        for (int tile = tile0; tile < num_tiles; tile += tile_step, ++it) {
          const int acc = it % C::ACC_STAGES;
          const uint32_t acc_phase = (it / C::ACC_STAGES) & 1;
          const int mb = m_block<CG>(p, tile, rank);
          const int m0 = mb * BLOCK_M + quarter * 32;
          const int n0 = (tile % p.n_tiles) * BLOCK_N;
          wait_acc(&tfull_bar[acc], acc_phase);
          tcgen05_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * C::ACC_COLS;
#pragma unroll 1
          for (int c = (mb < p.m_tiles ? half : CHUNKS); c < CHUNKS; c += 2) {
            uint32_t r[32];
            tmem_ld_chunk<32>(taddr + c * 32, r);
            if constexpr (NSPLIT == 2) {
              uint32_t r2[32];
              tmem_ld_chunk<32>(taddr + BLOCK_N + c * 32, r2);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
            } else {
              tmem_ld_wait();
            }
            const int n = n0 + c * 32;
            float v[32];
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 al = __ldg(reinterpret_cast<const float4*>(ep.alpha + n + j));
              const float4 be = __ldg(reinterpret_cast<const float4*>(ep.beta + n + j));
              v[j + 0] = fmaf(__uint_as_float(r[j + 0]), al.x, be.x);
              v[j + 1] = fmaf(__uint_as_float(r[j + 1]), al.y, be.y);
              v[j + 2] = fmaf(__uint_as_float(r[j + 2]), al.z, be.z);
              v[j + 3] = fmaf(__uint_as_float(r[j + 3]), al.w, be.w);
            }
            if (ep.relu) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            {
              float amax = 0.f;
#pragma unroll
              for (int j = 0; j < 32; ++j) amax = fmaxf(amax, fabsf(v[j]));
              flag_if_out_of_range(amax, ep.ovf);
            }
            // the staging buffer was handed to the TMA one chunk ago: wait until that store has read it
            if (leader) tma_store_wait_read<0>();
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 h, l;
              __half2* hh = reinterpret_cast<__half2*>(&h);
              __half2* ll = reinterpret_cast<__half2*>(&l);
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const __half2 hv = __floats2half2_rn(v[8 * j + 2 * t], v[8 * j + 2 * t + 1]);
                hh[t] = hv;
                const float2 hf = __half22float2(hv);
                ll[t] = __floats2half2_rn(v[8 * j + 2 * t] - hf.x, v[8 * j + 2 * t + 1] - hf.y);
              }
              *reinterpret_cast<uint4*>(buf + lane * 64 + ((j ^ swz) << 4)) = h;
              if constexpr (NSPLIT == 2) *reinterpret_cast<uint4*>(buf + C::STG_TILE_BYTES + lane * 64 + ((j ^ swz) << 4)) = l;
            }
            fence_proxy_async();
            __syncwarp();
            if (leader) {
#pragma unroll
              for (int s = 0; s < NSPLIT; ++s) tma_store_2d(&p.tmOut[s], buf + s * C::STG_TILE_BYTES, n, m0);
              tma_store_commit();
            }
          }
          tcgen05_fence_before();
          __syncwarp();
          if (leader) release_acc(acc);
        }
        if (leader) tma_store_wait_all();
        it = -1;   // tiles consumed
      }
    }
    for (int tile = tile0; it >= 0 && tile < num_tiles; tile += tile_step, ++it) {
      const int acc = it % C::ACC_STAGES;
      const uint32_t acc_phase = (it / C::ACC_STAGES) & 1;
      const int m0 = m_block<CG>(p, tile, rank) * BLOCK_M;
      const int n0 = (tile % p.n_tiles) * BLOCK_N;
      const int m = m0 + quarter * 32 + lane;
      const bool row_ok = m < p.M;
      wait_acc(&tfull_bar[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * C::ACC_COLS;
#pragma unroll 1
      for (int c0 = half * CH; c0 < BLOCK_N; c0 += 2 * CH) {
        uint32_t r[CH];
        tmem_ld_chunk<CH>(taddr + c0, r);
        if constexpr (NSPLIT == 2) {
          uint32_t r2[CH];
          tmem_ld_chunk<CH>(taddr + BLOCK_N + c0, r2);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < CH; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(r2[j]));
        } else {
          tmem_ld_wait();
        }
        const int n = n0 + c0;
        float v[CH];
#pragma unroll
        for (int j = 0; j < CH; j += 4) {
          const float4 al = __ldg(reinterpret_cast<const float4*>(ep.alpha + n + j));
          const float4 be = __ldg(reinterpret_cast<const float4*>(ep.beta + n + j));
          v[j + 0] = fmaf(__uint_as_float(r[j + 0]), al.x, be.x);
          v[j + 1] = fmaf(__uint_as_float(r[j + 1]), al.y, be.y);
          v[j + 2] = fmaf(__uint_as_float(r[j + 2]), al.z, be.z);
          v[j + 3] = fmaf(__uint_as_float(r[j + 3]), al.w, be.w);
        }
        if (row_ok) {
          if (ep.res_hi != nullptr) {
            const size_t off = static_cast<size_t>(m) * p.Cout + n;
#pragma unroll
            for (int j = 0; j < CH; j += 8) {
              const uint4 h = *reinterpret_cast<const uint4*>(ep.res_hi + off + j);
              const __half2* hh = reinterpret_cast<const __half2*>(&h);
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const float2 f = __half22float2(hh[t]);
                v[j + 2 * t] += f.x;
                v[j + 2 * t + 1] += f.y;
              }
              if (ep.res_lo != nullptr) {
                const uint4 l = *reinterpret_cast<const uint4*>(ep.res_lo + off + j);
                const __half2* ll = reinterpret_cast<const __half2*>(&l);
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                  const float2 f = __half22float2(ll[t]);
                  v[j + 2 * t] += f.x;
                  v[j + 2 * t + 1] += f.y;
                }
              }
            }
          }
          if (ep.relu) {
#pragma unroll
            for (int j = 0; j < CH; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          if (ep.out_mode == OUT_NHWC_SPLIT) {
            float amax = 0.f;
#pragma unroll
            for (int j = 0; j < CH; ++j) amax = fmaxf(amax, fabsf(v[j]));
            flag_if_out_of_range(amax, ep.ovf);
            const size_t off = static_cast<size_t>(m) * p.Cout + n;
#pragma unroll
            for (int j = 0; j < CH; j += 8) {
              uint4 h, l;
              __half2* hh = reinterpret_cast<__half2*>(&h);
              __half2* ll = reinterpret_cast<__half2*>(&l);
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                const __half2 hv = __floats2half2_rn(v[j + 2 * t], v[j + 2 * t + 1]);
                hh[t] = hv;
                const float2 hf = __half22float2(hv);
                ll[t] = __floats2half2_rn(v[j + 2 * t] - hf.x, v[j + 2 * t + 1] - hf.y);
              }
              *reinterpret_cast<uint4*>(ep.out_hi + off + j) = h;
              if (ep.out_lo != nullptr) *reinterpret_cast<uint4*>(ep.out_lo + off + j) = l;
            }
          } else if (ep.out_mode == OUT_NHWC_F32) {
            float* dst = ep.out_f32 + static_cast<size_t>(m) * p.Cout + n;
#pragma unroll
            for (int j = 0; j < CH; j += 4)
              *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {  // OUT_NCHW_F32: lanes are consecutive pixels of one image plane -> coalesced
            const int b = m / HoWo;
            const int hw = m - b * HoWo;
            float* dst = ep.out_f32 + (static_cast<size_t>(b) * p.Cout + n) * HoWo + hw;
            // write-once output: stream past L2.  The channel bound is warp-uniform: full chunks take the branch-free
            // path with a running pointer (a per-store bound check + 64-bit multiply cost ~17 instructions per store)
            if (n + CH <= p.Cout) {
#pragma unroll
              for (int j = 0; j < CH; ++j) {
                __stcs(dst, v[j]);
                dst += HoWo;
              }
            } else {
#pragma unroll
              for (int j = 0; j < CH; ++j) {
                if (n + j < p.Cout) __stcs(dst, v[j]);
                dst += HoWo;
              }
            }
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) release_acc(acc);
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();   // both CTAs are done with the pair's TMEM and with signalling each other
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    if constexpr (CG == 2) tmem_dealloc_pair<C::TMEM_COLS>(tmem_base);
    else tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------ host side: tensor maps
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
using EncodeIm2colFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct DriverApi {
  EncodeTiledFn tiled = nullptr;
  EncodeIm2colFn im2col = nullptr;
  int driver_version = 0;
};

// The driver entry points are resolved at run time so the library has no link-time libcuda
// dependency (it must load on a box without a GPU driver for the symbol-export test).
const DriverApi& driver_api() {
  static DriverApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    SMK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    SMK_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
    api.tiled = reinterpret_cast<EncodeTiledFn>(fn);
    fn = nullptr;
    SMK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
    SMK_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeIm2col not available");
    api.im2col = reinterpret_cast<EncodeIm2colFn>(fn);
    SMK_CUDA(cudaDriverGetVersion(&api.driver_version));
  });
  return api;
}

// Tensor-map cache.  cuTensorMapEncode* costs a few microseconds on the host and a launch needs up to eight maps; the
// engine's bump arenas hand out the same addresses every step, so the (pointer, geometry) key of every map repeats from
// the second step on.  Keyed by the encode arguments themselves, so a hit is exactly what the driver would build.
struct MapKey {
  uint64_t v[16];
  bool operator==(const MapKey& o) const { return std::memcmp(v, o.v, sizeof v) == 0; }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    uint64_t h = 0x9E3779B97F4A7C15ull;
    for (uint64_t x : k.v) { h ^= x + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2); }
    return (size_t)h;
  }
};
template <typename F>
CUtensorMap cached_map(const MapKey& key, F&& encode) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  int dev = 0;
  cudaGetDevice(&dev);
  MapKey k = key;
  k.v[15] = (uint64_t)dev;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(k);
  if (it != cache.end()) return it->second;
  if (cache.size() > 65536) cache.clear();             // unbounded callers (standalone ops on fresh buffers)
  CUtensorMap m = encode();
  cache.emplace(k, m);
  return m;
}

CUtensorMap make_map_2d_raw(const __half* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer) {
  CUtensorMap m;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {inner * sizeof(__half)};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  // operand tiles: the swizzle span equals the k-block row (64 fp16 = 128 B)
  CUresult r = driver_api().tiled(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides,
                                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SMK_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed, code " + std::to_string((int)r));
  return m;
}

CUtensorMap make_map_2d(const __half* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer) {
  MapKey k{};
  k.v[0] = 1; k.v[1] = (uint64_t)base; k.v[2] = inner; k.v[3] = outer; k.v[4] = box_inner; k.v[5] = box_outer;
  return cached_map(k, [&] { return make_map_2d_raw(base, inner, outer, box_inner, box_outer); });
}

CUtensorMap make_map_epilogue_raw(const __half* base, uint64_t cout, uint64_t m) {
  CUtensorMap t;
  cuuint64_t dims[2] = {cout, m};
  cuuint64_t strides[1] = {cout * sizeof(__half)};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = driver_api().tiled(&t, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides,
                                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SMK_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (epilogue) failed, code " + std::to_string((int)r));
  return t;
}

CUtensorMap make_map_epilogue(const __half* base, uint64_t cout, uint64_t m) {
  MapKey k{};
  k.v[0] = 2; k.v[1] = (uint64_t)base; k.v[2] = cout; k.v[3] = m;
  return cached_map(k, [&] { return make_map_epilogue_raw(base, cout, m); });
}

CUtensorMap make_map_im2col_raw(const __half* base, const Act& in, const ConvGeom& g) {
  CUtensorMap m;
  cuuint64_t dims[4] = {(cuuint64_t)in.C, (cuuint64_t)in.W, (cuuint64_t)in.H, (cuuint64_t)in.B};
  cuuint64_t strides[3] = {(cuuint64_t)in.C * 2, (cuuint64_t)in.W * in.C * 2, (cuuint64_t)in.H * in.W * in.C * 2};
  // fprop corners (cutlass/conv/collective/detail.hpp compute_{lower,upper}_corner_whd):
  //   lower = -pad, upper = pad - (k-1)*dilation; base pixel = lower + q*stride, tap offset = s*dilation.
  int lower[2] = {-g.pad, -g.pad};
  int upper[2] = {g.pad - (g.KW - 1) * g.dil, g.pad - (g.KH - 1) * g.dil};
  cuuint32_t estr[4] = {1, (cuuint32_t)g.stride, (cuuint32_t)g.stride, 1};
  const DriverApi& api = driver_api();
  CUresult r = api.im2col(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), dims, strides, lower,
                          upper, BLOCK_K, BLOCK_M, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SMK_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeIm2col failed, code " + std::to_string((int)r));
  // Same small-tensor descriptor fix-up CuTe applies for drivers <= 13.1
  // (cute/atom/copy_traits_sm90_im2col.hpp, make_im2col_tma_copy_desc).
  if (api.driver_version <= 13010 && in.numel() * sizeof(__half) < 131072)
    reinterpret_cast<uint64_t*>(&m)[1] &= ~(1ull << 21);
  return m;
}

CUtensorMap make_map_im2col(const __half* base, const Act& in, const ConvGeom& g) {
  MapKey k{};
  k.v[0] = 3; k.v[1] = (uint64_t)base;
  k.v[2] = ((uint64_t)in.B << 32) | (uint32_t)in.H; k.v[3] = ((uint64_t)in.W << 32) | (uint32_t)in.C;
  k.v[4] = ((uint64_t)g.KH << 32) | (uint32_t)g.KW; k.v[5] = ((uint64_t)g.stride << 32) | (uint32_t)g.pad;
  k.v[6] = (uint64_t)g.dil;
  return cached_map(k, [&] { return make_map_im2col_raw(base, in, g); });
}

template <int BLOCK_N, int NSPLIT, int CG = 1>
void launch_cfg(const GemmParams& p, int num_sms, cudaStream_t st) {
  using C = Cfg<BLOCK_N, NSPLIT, CG>;
  auto kern = conv_gemm_kernel<BLOCK_N, NSPLIT, CG>;
  static unsigned long long attr_done = 0;
  ensure_dynamic_smem(kern, C::SMEM_BYTES, attr_done);
  const int tiles = ((p.m_tiles + CG - 1) / CG) * p.n_tiles;
  const int slots = num_sms / CG;                      // one CTA (pair) per SM (pair)
  const int grid = (tiles < slots ? tiles : slots) * CG;
  if constexpr (CG == 1) {
    kern<<<grid, NUM_THREADS, C::SMEM_BYTES, st>>>(p);
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = CG;
    attr.val.clusterDim.y = 1;
    attr.val.clusterDim.z = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    SMK_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
  }
  SMK_CUDA(cudaGetLastError());
}

}  // namespace

// 2-D fp16 tensor map with a chosen swizzle span (32 / 64 / 128 bytes); shared with stem_sm100.cu
static CUtensorMap make_map_2d_any_raw(const __half* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer,
                            int swizzle_bytes) {
  CUtensorMap m;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {inner * sizeof(__half)};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = driver_api().tiled(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides,
                                  box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SMK_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed, code " + std::to_string((int)r));
  return m;
}

CUtensorMap make_map_2d_any(const __half* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer,
                            int swizzle_bytes) {
  MapKey k{};
  k.v[0] = 5; k.v[1] = (uint64_t)base; k.v[2] = inner; k.v[3] = outer; k.v[4] = box_inner; k.v[5] = box_outer;
  k.v[6] = (uint64_t)swizzle_bytes;
  return cached_map(k, [&] { return make_map_2d_any_raw(base, inner, outer, box_inner, box_outer, swizzle_bytes); });
}

// N-dimensional tiled-mode fp16 tensor map (rank 2..5), operand-load flavour (L2 promotion 256 B); shared with
// conv3x3_patch_sm100.cu
static CUtensorMap make_map_tiled_nd_raw(const __half* base, int rank, const uint64_t* dims,
                                         const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes) {
  SMK_CHECK(rank >= 2 && rank <= 5, "tensor map rank");
  CUtensorMap m;
  cuuint64_t d[5], sb[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) sb[i] = strides_bytes[i];
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = driver_api().tiled(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<__half*>(base), d, sb,
                                  bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SMK_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (nd) failed, code " + std::to_string((int)r));
  return m;
}

CUtensorMap make_map_tiled_nd(const __half* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                              const uint32_t* box, int swizzle_bytes) {
  SMK_CHECK(rank >= 2 && rank <= 5, "tensor map rank");
  MapKey k{};
  k.v[0] = 4 | ((uint64_t)rank << 8) | ((uint64_t)swizzle_bytes << 16);
  k.v[1] = (uint64_t)base;
  for (int i = 0; i < rank; ++i) k.v[2 + i] = dims[i] | ((uint64_t)box[i] << 40);
  for (int i = 0; i + 1 < rank; ++i) k.v[7 + i] = strides_bytes[i];
  return cached_map(k, [&] { return make_map_tiled_nd_raw(base, rank, dims, strides_bytes, box, swizzle_bytes); });
}

bool gemm_conv_supported(const ConvGeom& g) { return g.Cin % CIN_GRAIN == 0 && g.Cout >= 1; }

int gemm_cout_pad(int cout) {
  if (cout <= 16) return 16;
  if (cout <= 32) return 32;
  if (cout <= 64) return 64;
  if (cout <= 128) return 128;
  return (cout + 255) / 256 * 256;
}

void launch_gemm_conv(const Act& in, const ConvGeom& g, const __half* w_hi, const __half* w_lo, int cout_pad,
                      const Epilogue& ep, int nsplit, int num_sms, cudaStream_t st) {
  GemmInput gi{in, g, 0};
  launch_gemm_multi(&gi, 1, nullptr, -1, w_hi, w_lo, cout_pad, g.KH * g.KW * g.Cin, ep, nsplit, num_sms, st);
}

void launch_gemm_multi(const GemmInput* convs, int nconv, const Act* residual, int res_col0, const __half* w_hi,
                       const __half* w_lo, int cout_pad, int w_ld, const Epilogue& ep_in, int nsplit, int num_sms,
                       cudaStream_t st, bool reverse_m) {
  SMK_CHECK(nconv >= 1 && nconv <= 2, "1 or 2 convolution segments");
  SMK_CHECK(nconv + (residual != nullptr ? 1 : 0) <= 2, "at most two K segments");
  Epilogue ep = ep_in;
  const ConvGeom& g0 = convs[0].g;
  const Act& in0 = convs[0].in;
  const int Ho = g0.out_size(in0.H), Wo = g0.out_size(in0.W);
  GemmParams p;
  p.M = in0.B * Ho * Wo;
  p.Cout = g0.Cout;
  p.Ho = Ho;
  p.Wo = Wo;
  // Tile choice.  fast: 128 x min(Cout, 256), single CTA.  exact: 128 x min(Cout, 128) with two double-buffered TMEM
  // accumulator pairs, or — when the main loop is long enough to amortise a non-overlapped epilogue (>= kPairMinKb
  // k-blocks) — a 256 x 256 CTA-pair tile with a single accumulator stage.  The SM's shared-memory port (128 B/clk)
  // carries both the TMA fills and the operand reads of every tcgen05.mma; per k-block a 128 x 128 exact tile moves
  // 64 KB in + 96 KB out of smem for 768 MMA-clocks (208 B/clk -> <= 61 % tensor duty, 63-66 % measured), a 128 x 256
  // tile 96 + 144 KB for 1536 (156 B/clk -> <= 82 %).  Measured on B200 (profiles/r01_tile_ab.md): layer3.0
  // conv3+downsample 1.45 -> 1.16 ms, 3x3 convs -10..-17 %, short-K 1x1 layers +8..+35 % slower (they stay on
  // 128 x 128).  32-wide k-blocks (64 B rows) were slower everywhere.
  // A CTA pair (cluster of 2, tcgen05 cta_group::2) stages its own 128 A rows per CTA and half of the B rows, so fills
  // and operand reads through the smem port drop by a third (104 B/clk for the exact 256-wide tile).  Measured
  // (profiles/r01_tile_ab.md): exact long-K layers -4..-9 %; fast 256-wide pairs +5..+12 % slower (not smem-bound);
  // 256 x 128 pairs on the short-K exact layers neutral to slower (lock-step epilogues).
  // The wide tile is taken only when the 128 x 128 tiling fills the machine anyway (small batches — B=1: 64 tiles —
  // are latency bound and want as many CTAs as they can get), and only for NHWC split outputs: the 3969-channel NCHW
  // mask head (K = 256) is slower on wide or pair tiles, its scalar-store epilogue needs the overlap (DESIGN.md §8).
  constexpr int kPairMinKb = 24;
  int total_kb = residual != nullptr ? 2 : 0;
  for (int i = 0; i < nconv; ++i) total_kb += convs[i].g.KH * convs[i].g.KW * convs[i].g.Cin / BLOCK_K;
  const long long narrow_tiles = (long long)((p.M + BLOCK_M - 1) / BLOCK_M) * (cout_pad / 128);
  const bool pair = nsplit == 2 && cout_pad >= 256 && ep.out_mode == OUT_NHWC_SPLIT && total_kb >= kPairMinKb &&
                    narrow_tiles >= num_sms;
  const int block_n = pair ? 256 : std::min(cout_pad, nsplit == 2 ? 128 : 256);
  const int cg = pair ? 2 : 1;
  SMK_CHECK(cout_pad % block_n == 0, "cout_pad must be a multiple of the N tile");
  if (ep.out_mode != OUT_NCHW_F32) SMK_CHECK(g0.Cout == cout_pad, "NHWC outputs need Cout to match the padded tile width");
  p.n_tiles = cout_pad / block_n;
  p.m_tiles = (p.M + BLOCK_M - 1) / BLOCK_M;
  p.reverse_m = reverse_m ? 1 : 0;
  p.nseg = 0;
  for (int i = 0; i < nconv; ++i) {
    const ConvGeom& g = convs[i].g;
    const Act& in = convs[i].in;
    SMK_CHECK(gemm_conv_supported(g), "Cin must be a multiple of 64 for the tensor-core conv");
    SMK_CHECK(in.C == g.Cin && g.Cout == g0.Cout && in.B == in0.B, "segment channels/batch mismatch");
    SMK_CHECK(g.out_size(in.H) == Ho && g.out_size(in.W) == Wo, "segments must produce the same output size");
    SMK_CHECK(nsplit == 1 || (in.lo != nullptr && w_lo != nullptr), "exact mode needs lo planes");
    GemmSegment& sg = p.seg[p.nseg++];
    sg.kind = 0;
    sg.cblks = g.Cin / BLOCK_K;
    sg.num_kb = g.KH * g.KW * sg.cblks;
    sg.KW = g.KW;
    sg.stride = g.stride;
    sg.pad = g.pad;
    sg.dil = g.dil;
    sg.mode = (g.KH == 1 && g.KW == 1 && g.stride == 1 && g.pad == 0) ? 0 : 1;
    sg.b_col0 = convs[i].w_col0;
    SMK_CHECK(sg.b_col0 % 64 == 0 && sg.b_col0 + g.KH * g.KW * g.Cin <= w_ld, "weight column range");
    for (int s = 0; s < nsplit; ++s) {
      const __half* a = s == 0 ? in.hi : in.lo;
      sg.tmA[s] = sg.mode == 0 ? make_map_2d(a, g.Cin, (uint64_t)in.M(), BLOCK_K, BLOCK_M) : make_map_im2col(a, in, g);
    }
    if (nsplit == 1) sg.tmA[1] = sg.tmA[0];
  }
  if (residual != nullptr) {
    // the residual rides the tensor pipe: needs the diag(2^e) block in the weights and 64-wide column blocks
    SMK_CHECK(res_col0 >= 0 && res_col0 % 64 == 0 && res_col0 + g0.Cout <= w_ld && block_n % 64 == 0,
              "identity segment needs a diagonal block in the packed weights");
    SMK_CHECK(residual->C == g0.Cout && residual->M() == p.M, "residual shape");
    SMK_CHECK(nsplit == 1 || residual->lo != nullptr, "exact mode residual needs both planes");
    GemmSegment& sg = p.seg[p.nseg++];
    sg.kind = 1;
    sg.mode = 0;
    sg.num_kb = block_n / BLOCK_K;
    sg.cblks = sg.KW = sg.stride = sg.dil = 1;
    sg.pad = 0;
    sg.b_col0 = res_col0;
    for (int s = 0; s < nsplit; ++s)
      sg.tmA[s] = make_map_2d(s == 0 ? residual->hi : residual->lo, g0.Cout, (uint64_t)p.M, BLOCK_K, BLOCK_M);
    if (nsplit == 1) sg.tmA[1] = sg.tmA[0];
    ep.res_hi = ep.res_lo = nullptr;       // accumulated by the MMA, not by the epilogue
  }
  if (p.nseg == 1) p.seg[1] = p.seg[0];
  for (int s = 0; s < nsplit; ++s)
    p.tmB[s] = make_map_2d(s == 0 ? w_hi : w_lo, (uint64_t)w_ld, cout_pad, BLOCK_K, block_n / cg);
  if (nsplit == 1) p.tmB[1] = p.tmB[0];
  // NHWC split outputs go through smem + TMA stores; an epilogue-side residual (no diagonal block) needs the
  // direct path
  p.staged = (ep.out_mode == OUT_NHWC_SPLIT && block_n >= 32 && g0.Cout % 32 == 0 && ep.res_hi == nullptr) ? 1 : 0;
  if (p.staged) {
    SMK_CHECK(nsplit == 1 || ep.out_lo != nullptr, "exact mode writes both planes");
    for (int s = 0; s < nsplit; ++s) p.tmOut[s] = make_map_epilogue(s == 0 ? ep.out_hi : ep.out_lo, g0.Cout, p.M);
    if (nsplit == 1) p.tmOut[1] = p.tmOut[0];
  } else {
    p.tmOut[0] = p.tmOut[1] = p.tmB[0];
  }
  p.ep = ep;

#define SMK_DISPATCH(BN)                                             \
  case BN:                                                           \
    if (nsplit == 2) launch_cfg<BN, 2>(p, num_sms, st);              \
    else launch_cfg<BN, 1>(p, num_sms, st);                          \
    break;
  switch (block_n) {
    SMK_DISPATCH(16)
    SMK_DISPATCH(32)
    SMK_DISPATCH(64)
    SMK_DISPATCH(128)
    case 256:   // exact mode reaches the 256-wide tile only as a CTA pair
      if (nsplit == 2) launch_cfg<256, 2, 2>(p, num_sms, st);
      else launch_cfg<256, 1>(p, num_sms, st);
      break;
    default: SMK_CHECK(false, "unsupported N tile");
  }
#undef SMK_DISPATCH
}

}  // namespace smk
