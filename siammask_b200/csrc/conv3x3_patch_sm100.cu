// 3x3 / stride 1 / pad 1 convolution with Cin = Cout = CM (64 or 128) — the conv2 of the layer1 / layer2 bottlenecks
// (resnet.py:66-76) — on tcgen05 WITHOUT im2col traffic.
//
// The general kernel (conv_gemm_sm100.cu) fetches every k-block of A with an im2col-mode TMA: each input pixel is
// pulled from L2 nine times (once per filter tap) as 128-byte rows, and at N = 64..128 output channels the TMA unit's
// row rate (~7 clk per 128-B im2col row, r01 launch list) — not the tensor pipe — paces the layer (layer1 conv2:
// 16 k clk per 128-pixel tile for 3.5 k clk of MMA).  Here a tile is RO whole image rows and its input PATCH
// (RO+2 rows x PW pixels x 64 channels per k-block, PW = W+1 rounded up to 8) is loaded ONCE by a tiled-mode 4-D TMA
// box starting at x = -1, y = y0-1: out-of-image pixels arrive as zeros, so in shared memory the patch is the
// zero-padded image in "padded-linear" form, row index = yy*PW + xx, where the column x = -1 of one image row doubles
// as the column x = W of the row above.  In that form EVERY filter tap is a constant row shift: output pixel j reads
// patch row j + r*PW + s - 1, so the nine taps are nine UMMA descriptors onto the same resident patch whose start
// address moves by (r*PW + s - 1) rows of 128 B (r*PW is a multiple of 8 rows = one swizzle atom; s - 1 in {-1,0,+1}
// shifts by single rows inside the 128B-swizzle pattern, which works because the pattern is a function of the
// shared-memory ADDRESS bits — the same reason advancing a descriptor by 32 B along K works).  Only the weights
// stream through a TMA ring (one 2-D tile per tap and k-block).
//
// Output rows of a tile are the PW-strided pixels (j % PW == 0 is the phantom column x = -1, never stored): with
// W = 63 / 31 / 15 and PW = 64 / 32 / 16 the waste is 1/PW.  Epilogue: TMEM -> registers -> affine (+ReLU) -> split fp16
// planes, stored straight to global (each thread owns one pixel = 2*CM contiguous bytes per plane).
//
// Warp roles as in conv_gemm_sm100.cu: warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2..9 = epilogue.
#include "common.cuh"
#include "ptx.cuh"

namespace smk {

namespace {

constexpr int P_THREADS = 320;
constexpr int P_SLACK_ROWS = 8;            // zeroed rows before and after every patch panel

template <int CM, int NSPLIT>
struct PCfg {
  static constexpr int NKB = CM / 64;                         // 64-channel k-blocks
  static constexpr int B_TILE_BYTES = CM * 128;               // one plane of one (tap, k-block) weight tile
  static constexpr int B_STAGE_BYTES = NSPLIT * B_TILE_BYTES;
  static constexpr int B_STAGES = 3;
  static constexpr int ACC_COLS = NSPLIT * CM;                // hi*hi accumulator + cross-term accumulator
  static constexpr int TMEM_COLS = 2 * ACC_COLS <= 256 ? 256 : 512;
  static_assert(2 * ACC_COLS <= 512, "two accumulator stages must fit TMEM");
};

struct PatchParams {
  CUtensorMap tmA[2];      // hi / lo input planes, 4-D (C, W, H, B), box (64, PW, RO+2, 1), 128B swizzle
  CUtensorMap tmB[2];      // hi / lo weights [CM][9*CM] K-major, box (64, CM)
  int B, H, W, PW, RO;
  int tiles_per_img, num_tiles;
  int panel_bytes;         // one plane of one patch buffer incl. slack rows
  int patch_rows;          // (RO+2)*PW
  Epilogue ep;
};

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// K-major SWIZZLE_128B descriptors: the start may sit on ANY 128-byte row of the swizzle pattern with the
// descriptor's base_offset field left 0 — measured on B200 (tests/test_gpu_ops.py, cases 3x3_p1*): the hardware applies
// the XOR to the shared-memory address bits, so a row shift needs no correction (setting base_offset = (addr >> 7) & 7,
// as the PTX text suggests for unaligned starts, gives wrong results).

template <int CM, int NSPLIT>
__global__ void __launch_bounds__(P_THREADS, 1) conv3x3_patch_kernel(const __grid_constant__ PatchParams p) {
  using C = PCfg<CM, NSPLIT>;
  constexpr int NKB = C::NKB;
  constexpr uint32_t idesc = umma_idesc_f16(128, CM);
  constexpr uint32_t idesc_cat = umma_idesc_f16(128, NSPLIT == 2 ? 2 * CM : CM);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  // layout: patch buffer 0 | patch buffer 1 (each NSPLIT panels) | B ring | barriers
  const int patch_bytes = NSPLIT * p.panel_bytes;
  uint8_t* bring = smem + 2 * patch_bytes;
  uint64_t* pfull = reinterpret_cast<uint64_t*>(bring + C::B_STAGES * C::B_STAGE_BYTES);
  uint64_t* pempty = pfull + 2;
  uint64_t* bfull = pempty + 2;
  uint64_t* bempty = bfull + C::B_STAGES;
  uint64_t* tfull = bempty + C::B_STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  // warp index through a shuffle: provably warp-uniform for the compiler (role branches stay convergent)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  // zero the slack rows around every panel once (TMA never writes them)
  {
    const int slack = P_SLACK_ROWS * 128;
    for (int pb = 0; pb < 2 * NSPLIT; ++pb) {
      uint8_t* panel = smem + pb * p.panel_bytes;
      for (int i = threadIdx.x * 16; i < 2 * slack; i += P_THREADS * 16) {
        uint8_t* dst = i < slack ? panel + i : panel + slack + p.patch_rows * 128 + (i - slack);
        *reinterpret_cast<uint4*>(dst) = make_uint4(0, 0, 0, 0);
      }
    }
    fence_proxy_async();
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < NSPLIT; ++i) { tma_prefetch_desc(&p.tmA[i]); tma_prefetch_desc(&p.tmB[i]); }
    for (int i = 0; i < 2; ++i) { mbar_init(&pfull[i], 1); mbar_init(&pempty[i], 1); }
    for (int i = 0; i < C::B_STAGES; ++i) { mbar_init(&bfull[i], 1); mbar_init(&bempty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 8); }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 1) {
    __syncwarp();
    tmem_alloc<C::TMEM_COLS>(tmem_slot);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  // broadcast through a shuffle so the compiler KNOWS the TMEM base is warp-uniform: tcgen05 operands live in uniform
  // registers, and a value that merely came out of shared memory makes ptxas wrap every single MMA in a
  // divergence ("waterfall") loop — ELECT / R2UR / branch per instruction, ~90 clk of issue time per MMA
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const int slack_bytes = P_SLACK_ROWS * 128;

  if (warp == 0) {
    // ===================== TMA producer (whole warp walks the loop, one elected lane issues) =====================
    const bool leader = elect_one();
    // units = (tile, k-block) pairs of this CTA in execution order; unit u uses patch buffer u & 1.  The patch of unit
    // u+1 is requested early in unit u (after as many weight tiles as the ring holds, so that waiting for its buffer —
    // freed when unit u-1 retires — never delays the first taps of unit u): it has most of a unit of MMAs to arrive.
    const int my_tiles = (p.num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int units = my_tiles * NKB;
    auto issue_patch = [&](int u) {
      const int tile = blockIdx.x + (u / NKB) * gridDim.x;
      const int kb = u % NKB;
      const int b = tile / p.tiles_per_img;
      const int y0 = (tile - b * p.tiles_per_img) * p.RO;
      const int pbuf = u & 1;
      const uint32_t pph = (u >> 1) & 1;
      mbar_wait_guarded(&pempty[pbuf], pph ^ 1);
      if (leader) {
        mbar_arrive_expect_tx(&pfull[pbuf], NSPLIT * p.patch_rows * 128);
#pragma unroll
        for (int s = 0; s < NSPLIT; ++s)
          tma_load_4d(smem + (pbuf * NSPLIT + s) * p.panel_bytes + slack_bytes, &p.tmA[s], &pfull[pbuf], kb * 64, -1,
                      y0 - 1, b);
      }
      __syncwarp();
    };
    int bstage = 0;
    uint32_t bphase = 0;
    if (units > 0) issue_patch(0);
    for (int u = 0; u < units; ++u) {
      const int kb = u % NKB;
      for (int tap = 0; tap < 9; ++tap) {
        if (tap == C::B_STAGES && u + 1 < units) issue_patch(u + 1);
        mbar_wait_guarded(&bempty[bstage], bphase ^ 1);
        if (leader) {
          mbar_arrive_expect_tx(&bfull[bstage], C::B_STAGE_BYTES);
          uint8_t* st = bring + bstage * C::B_STAGE_BYTES;
#pragma unroll
          for (int s = 0; s < NSPLIT; ++s)
            tma_load_2d(st + s * C::B_TILE_BYTES, &p.tmB[s], &bfull[bstage], tap * CM + kb * 64, 0);
        }
        __syncwarp();
        if (++bstage == C::B_STAGES) { bstage = 0; bphase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The WHOLE warp walks the loop (convergent control flow, all operands provably uniform) and one elected lane issues:
    // a `threadIdx.x == 32` branch makes ptxas wrap every tcgen05 instruction in a divergence loop.  Descriptors are
    // built once per tap; the K steps only add 32 B (>> 4) to their address fields.
    const bool leader = elect_one();
    int unit = 0, bstage = 0, it = 0;
    uint32_t bphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait_guarded(&tempty[acc], acc_phase ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + acc * C::ACC_COLS;
      uint32_t acc_main = 0;
      for (int kb = 0; kb < NKB; ++kb, ++unit) {
        const int pbuf = unit & 1;
        const uint32_t pph = (unit >> 1) & 1;
        mbar_wait_guarded(&pfull[pbuf], pph);
        tcgen05_fence_after();
        const uint32_t a_hi0 = smem_u32(smem + (pbuf * NSPLIT) * p.panel_bytes + slack_bytes);
        const uint32_t a_lo0 = a_hi0 + p.panel_bytes;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
          const int r = tap / 3, s = tap - 3 * r;
          const int shift = (r * p.PW + s - 1) * 128;           // bytes: patch row of output pixel 0 for this tap
          mbar_wait_guarded(&bfull[bstage], bphase);
          tcgen05_fence_after();
          const uint32_t b_hi = smem_u32(bring + bstage * C::B_STAGE_BYTES);
          const uint64_t da_hi = umma_desc_kmajor_sw128(a_hi0 + shift);
          const uint64_t da_lo = umma_desc_kmajor_sw128(a_lo0 + shift);
          const uint64_t db_hi = umma_desc_kmajor_sw128(b_hi);
          if (leader) {
            // exact mode: the lo weight tile follows the hi tile in the stage and the accumulators are adjacent TMEM
            // columns, so hi*hi and hi*lo are ONE MMA of N = 2*CM over [B_hi; B_lo] and the shifted A_hi view crosses
            // the smem port once for both (see conv_gemm_sm100.cu)
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t kadd = static_cast<uint64_t>(k * 2);   // 32 bytes >> 4 in the start-address field
              umma_f16(tmem_d, da_hi + kadd, db_hi + kadd, idesc_cat, acc_main);
              acc_main = 1;
              if constexpr (NSPLIT == 2) umma_f16(tmem_d + CM, da_lo + kadd, db_hi + kadd, idesc, 1u);
            }
            umma_commit(&bempty[bstage]);
            if (tap == 8) {
              umma_commit(&pempty[pbuf]);                          // patch buffer free once these MMAs retire
              if (kb == NKB - 1) umma_commit(&tfull[acc]);
            }
          }
          __syncwarp();
          acc_main = 1;
          if (++bstage == C::B_STAGES) { bstage = 0; bphase ^= 1; }
        }
      }
    }
  } else if (warp >= 2) {
    // ===================== epilogue =====================
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;                 // column half of the tile this warp converts
    constexpr int COLS_PER_WARP = CM / 2;
    const Epilogue& ep = p.ep;
    int it = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int b = tile / p.tiles_per_img;
      const int y0 = (tile - b * p.tiles_per_img) * p.RO;
      const int j = quarter * 32 + lane;              // tile row = padded-linear pixel
      const int yy = j / p.PW, xx = j - yy * p.PW;
      const int y = y0 + yy, x = xx - 1;
      const bool ok = x >= 0 && x < p.W && y < p.H && yy < p.RO;
      mbar_wait_guarded(&tfull[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * C::ACC_COLS;
      const size_t off0 = ((static_cast<size_t>(b) * p.H + y) * p.W + x) * CM;
#pragma unroll 1
      for (int c0 = half * COLS_PER_WARP; c0 < (half + 1) * COLS_PER_WARP; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + c0, r);
        if constexpr (NSPLIT == 2) {
          uint32_t r2[32];
          tmem_ld_32x32b_x32(taddr + CM + c0, r2);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 32; ++q) r[q] = __float_as_uint(__uint_as_float(r[q]) + __uint_as_float(r2[q]));
        } else {
          tmem_ld_wait();
        }
        float v[32];
#pragma unroll
        for (int q = 0; q < 32; q += 4) {
          const float4 al = __ldg(reinterpret_cast<const float4*>(ep.alpha + c0 + q));
          const float4 be = __ldg(reinterpret_cast<const float4*>(ep.beta + c0 + q));
          v[q + 0] = fmaf(__uint_as_float(r[q + 0]), al.x, be.x);
          v[q + 1] = fmaf(__uint_as_float(r[q + 1]), al.y, be.y);
          v[q + 2] = fmaf(__uint_as_float(r[q + 2]), al.z, be.z);
          v[q + 3] = fmaf(__uint_as_float(r[q + 3]), al.w, be.w);
        }
        if (ep.relu) {
#pragma unroll
          for (int q = 0; q < 32; ++q) v[q] = fmaxf(v[q], 0.f);
        }
        if (ok) {
          float amax = 0.f;
#pragma unroll
          for (int q = 0; q < 32; ++q) amax = fmaxf(amax, fabsf(v[q]));
          flag_if_out_of_range(amax, ep.ovf);
#pragma unroll
          for (int q = 0; q < 32; q += 8) {
            uint4 h, l;
            __half2* hh = reinterpret_cast<__half2*>(&h);
            __half2* ll = reinterpret_cast<__half2*>(&l);
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const __half2 hv = __floats2half2_rn(v[q + 2 * t], v[q + 2 * t + 1]);
              hh[t] = hv;
              const float2 hf = __half22float2(hv);
              ll[t] = __floats2half2_rn(v[q + 2 * t] - hf.x, v[q + 2 * t + 1] - hf.y);
            }
            *reinterpret_cast<uint4*>(ep.out_hi + off0 + c0 + q) = h;
            if (ep.out_lo != nullptr) *reinterpret_cast<uint4*>(ep.out_lo + off0 + c0 + q) = l;
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

int patch_pw(int W) { return (W + 1 + 7) / 8 * 8; }

// RO = image rows per 128-pixel tile
int patch_ro(int W) {
  const int pw = patch_pw(W);
  return 128 % pw == 0 ? 128 / pw : 0;
}

template <int CM, int NSPLIT>
void launch_patch(const PatchParams& p, int num_sms, cudaStream_t st) {
  using C = PCfg<CM, NSPLIT>;
  const int smem = 2 * NSPLIT * p.panel_bytes + C::B_STAGES * C::B_STAGE_BYTES + 256 + 1024;
  SMK_CHECK(smem <= 227 * 1024, "patch conv: shared memory budget");
  auto kern = conv3x3_patch_kernel<CM, NSPLIT>;
  static unsigned long long attr = 0;
  ensure_dynamic_smem(kern, 227 * 1024, attr);
  const int grid = p.num_tiles < num_sms ? p.num_tiles : num_sms;
  kern<<<grid, P_THREADS, smem, st>>>(p);
  SMK_CUDA(cudaGetLastError());
}

}  // namespace

bool patch_conv_supported(const Act& in, const ConvGeom& g) {
  if (!(g.KH == 3 && g.KW == 3 && g.stride == 1 && g.pad == 1 && g.dil == 1 && g.Cin == g.Cout)) return false;
  if (!(g.Cin == 64 || g.Cin == 128)) return false;
  if (in.H != in.W) return false;
  return patch_ro(in.W) >= 1 && patch_pw(in.W) <= 64;
}

void launch_conv3x3_patch(const Act& in, const ConvGeom& g, const __half* w_hi, const __half* w_lo, int w_ld,
                          const Epilogue& ep, int nsplit, int num_sms, cudaStream_t st) {
  SMK_CHECK(patch_conv_supported(in, g), "patch conv: unsupported geometry");
  SMK_CHECK(ep.out_mode == OUT_NHWC_SPLIT && ep.res_hi == nullptr, "patch conv writes NHWC split planes, no residual");
  SMK_CHECK(nsplit == 1 || (in.lo != nullptr && w_lo != nullptr && ep.out_lo != nullptr), "exact mode needs lo planes");
  SMK_CHECK(w_ld >= 9 * g.Cin, "weight row length");
  PatchParams p;
  p.B = in.B; p.H = in.H; p.W = in.W;
  p.PW = patch_pw(in.W);
  p.RO = patch_ro(in.W);
  p.tiles_per_img = (in.H + p.RO - 1) / p.RO;
  p.num_tiles = in.B * p.tiles_per_img;
  p.patch_rows = (p.RO + 2) * p.PW;
  p.panel_bytes = (p.patch_rows + 2 * P_SLACK_ROWS) * 128;
  SMK_CHECK(p.panel_bytes % 1024 == 0, "patch panels must keep the 1024-byte swizzle alignment");
  p.ep = ep;
  for (int s = 0; s < nsplit; ++s) {
    const __half* a = s == 0 ? in.hi : in.lo;
    const uint64_t dims[4] = {(uint64_t)in.C, (uint64_t)in.W, (uint64_t)in.H, (uint64_t)in.B};
    const uint64_t strides[3] = {(uint64_t)in.C * 2, (uint64_t)in.W * in.C * 2, (uint64_t)in.H * in.W * in.C * 2};
    const uint32_t box[4] = {64, (uint32_t)p.PW, (uint32_t)(p.RO + 2), 1};
    p.tmA[s] = make_map_tiled_nd(a, 4, dims, strides, box, 128);
    const uint64_t wd[2] = {(uint64_t)w_ld, (uint64_t)g.Cout};
    const uint64_t ws[1] = {(uint64_t)w_ld * 2};
    const uint32_t wb[2] = {64, (uint32_t)g.Cout};
    p.tmB[s] = make_map_tiled_nd(s == 0 ? w_hi : w_lo, 2, wd, ws, wb, 128);
  }
  if (nsplit == 1) { p.tmA[1] = p.tmA[0]; p.tmB[1] = p.tmB[0]; }
  if (g.Cin == 64) {
    if (nsplit == 2) launch_patch<64, 2>(p, num_sms, st); else launch_patch<64, 1>(p, num_sms, st);
  } else {
    if (nsplit == 2) launch_patch<128, 2>(p, num_sms, st); else launch_patch<128, 1>(p, num_sms, st);
  }
}

}  // namespace smk
