// CUDA-core kernels of the SiamMask hot path (sm_100a): everything that is not a dense contraction
// large enough for the tensor pipe — the 3-channel 7x7 stem, max-pool, the bandwidth-bound depthwise
// cross-correlation, the crops/gathers of the refine stage, its 1-32 channel 3x3 convs and the
// 1x1 -> 15x15 transposed conv — plus a plain reference convolution used to bisect the tcgen05 path.
#include "common.cuh"

#include <cmath>
#include <type_traits>
#include <cstdlib>
#include <vector>

namespace smk {

namespace {

__device__ __forceinline__ float split_load(const __half* hi, const __half* lo, size_t i) {
  float v = __half2float(hi[i]);
  if (lo != nullptr) v += __half2float(lo[i]);
  return v;
}
__device__ __forceinline__ void split_store(__half* hi, __half* lo, size_t i, float v) {
  const __half h = __float2half_rn(v);
  hi[i] = h;
  if (lo != nullptr) lo[i] = __float2half_rn(v - __half2float(h));
}
__device__ __forceinline__ void split_store2(__half* hi, __half* lo, size_t i, float2 v) {
  const __half2 h = __floats2half2_rn(v.x, v.y);
  *reinterpret_cast<__half2*>(hi + i) = h;
  if (lo != nullptr) {
    const float2 hf = __half22float2(h);
    *reinterpret_cast<__half2*>(lo + i) = __floats2half2_rn(v.x - hf.x, v.y - hf.y);
  }
}

// ------------------------------------------------------------------------------------------------
// Reference convolution (one thread per output element, fp32 accumulate).  Same epilogue contract
// as the tensor-core kernel.  Weights: fp32 [KH][KW][Cin][Cout].
__global__ void ref_conv_kernel(Act in, ConvGeom g, const float* __restrict__ w, Epilogue ep, int Ho, int Wo) {
  const size_t total = (size_t)in.B * Ho * Wo * g.Cout;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int n = idx % g.Cout;
    const size_t m = idx / g.Cout;
    const int wo = m % Wo;
    const int ho = (m / Wo) % Ho;
    const int b = m / ((size_t)Wo * Ho);
    float acc = 0.f;
    for (int r = 0; r < g.KH; ++r) {
      const int hi_ = ho * g.stride - g.pad + r * g.dil;
      if (hi_ < 0 || hi_ >= in.H) continue;
      for (int s = 0; s < g.KW; ++s) {
        const int wi = wo * g.stride - g.pad + s * g.dil;
        if (wi < 0 || wi >= in.W) continue;
        const size_t ibase = (((size_t)b * in.H + hi_) * in.W + wi) * in.C;
        const float* wp = w + ((size_t)(r * g.KW + s) * g.Cin) * g.Cout + n;
        for (int c = 0; c < g.Cin; ++c) acc = fmaf(split_load(in.hi, in.lo, ibase + c), wp[(size_t)c * g.Cout], acc);
      }
    }
    float v = fmaf(acc, ep.alpha[n], ep.beta[n]);
    if (ep.res_hi != nullptr) v += split_load(ep.res_hi, ep.res_lo, m * g.Cout + n);
    if (ep.relu) v = fmaxf(v, 0.f);
    if (ep.out_mode == OUT_NHWC_SPLIT) split_store(ep.out_hi, ep.out_lo, m * g.Cout + n, v);
    else if (ep.out_mode == OUT_NHWC_F32) ep.out_f32[m * g.Cout + n] = v;
    else ep.out_f32[((size_t)b * g.Cout + n) * Ho * Wo + (size_t)ho * Wo + wo] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// Stem: 7x7 stride-2 pad-0 conv, 3 -> 64 channels, + BN + ReLU (resnet.py:154,218-220).
// Input: raw NCHW fp32 pixels (the boundary layout, tools/test.py:61-64); output: p0, NHWC split planes.
// Block = 16x8 output pixels x 64 channels; thread = 2 horizontally adjacent pixels x 16 channels.
constexpr int ST_TW = 16, ST_TH = 8, ST_PW = ST_TW * 2 + 5, ST_PH = ST_TH * 2 + 5;

__global__ void __launch_bounds__(256) stem_kernel(const float* __restrict__ x, int S, int So,
                                                   const float* __restrict__ w,      // [7][7][3][64]
                                                   const float* __restrict__ alpha, const float* __restrict__ beta,
                                                   Act out) {
  __shared__ __align__(16) float sw[147 * 64];
  __shared__ float sp[3][ST_PH][ST_PW];
  const int b = blockIdx.z;
  const int oy0 = blockIdx.y * ST_TH, ox0 = blockIdx.x * ST_TW;
  for (int i = threadIdx.x; i < 147 * 64; i += 256) sw[i] = w[i];
  const float* xb = x + (size_t)b * 3 * S * S;
  for (int i = threadIdx.x; i < 3 * ST_PH * ST_PW; i += 256) {
    const int c = i / (ST_PH * ST_PW);
    const int rem = i - c * (ST_PH * ST_PW);
    const int py = rem / ST_PW, px = rem - py * ST_PW;
    const int iy = oy0 * 2 + py, ix = ox0 * 2 + px;
    sp[c][py][px] = (iy < S && ix < S) ? xb[((size_t)c * S + iy) * S + ix] : 0.f;
  }
  __syncthreads();
  const int cg = threadIdx.x >> 6;          // channel group of 16 (warp-uniform)
  const int pp = threadIdx.x & 63;          // pixel pair
  const int ty = pp >> 3, tx = (pp & 7) * 2;
  float acc0[16], acc1[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) { acc0[j] = 0.f; acc1[j] = 0.f; }
  for (int r = 0; r < 7; ++r) {
    for (int s = 0; s < 7; ++s) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float a0 = sp[c][ty * 2 + r][tx * 2 + s];
        const float a1 = sp[c][ty * 2 + r][tx * 2 + 2 + s];
        const float4* wv = reinterpret_cast<const float4*>(&sw[((r * 7 + s) * 3 + c) * 64 + cg * 16]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 q = wv[j];
          acc0[4 * j + 0] = fmaf(a0, q.x, acc0[4 * j + 0]); acc1[4 * j + 0] = fmaf(a1, q.x, acc1[4 * j + 0]);
          acc0[4 * j + 1] = fmaf(a0, q.y, acc0[4 * j + 1]); acc1[4 * j + 1] = fmaf(a1, q.y, acc1[4 * j + 1]);
          acc0[4 * j + 2] = fmaf(a0, q.z, acc0[4 * j + 2]); acc1[4 * j + 2] = fmaf(a1, q.z, acc1[4 * j + 2]);
          acc0[4 * j + 3] = fmaf(a0, q.w, acc0[4 * j + 3]); acc1[4 * j + 3] = fmaf(a1, q.w, acc1[4 * j + 3]);
        }
      }
    }
  }
  const int oy = oy0 + ty;
#pragma unroll
  for (int px = 0; px < 2; ++px) {
    const int ox = ox0 + tx + px;
    if (oy >= So || ox >= So) continue;
    const float* acc = px == 0 ? acc0 : acc1;
    const size_t base = (((size_t)b * So + oy) * So + ox) * 64 + cg * 16;
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
      float2 v;
      v.x = fmaxf(fmaf(acc[j], alpha[cg * 16 + j], beta[cg * 16 + j]), 0.f);
      v.y = fmaxf(fmaf(acc[j + 1], alpha[cg * 16 + j + 1], beta[cg * 16 + j + 1]), 0.f);
      split_store2(out.hi, out.lo, base + j, v);
    }
  }
}

// 3x3 stride-2 pad-1 max-pool over NHWC split planes (resnet.py:158,221); thread = pixel x 8 channels
// (one 16-byte load per plane and tap).
__global__ void maxpool_kernel(Act in, Act out) {
  const size_t total = out.numel() / 8;
  const int c8n = out.C / 8;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int c = (idx % c8n) * 8;
    const size_t m = idx / c8n;
    const int wo = m % out.W, ho = (m / out.W) % out.H;
    const int b = m / ((size_t)out.W * out.H);
    float best[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) best[j] = -INFINITY;
    for (int r = 0; r < 3; ++r) {
      const int hi_ = ho * 2 - 1 + r;
      if (hi_ < 0 || hi_ >= in.H) continue;
      for (int s = 0; s < 3; ++s) {
        const int wi = wo * 2 - 1 + s;
        if (wi < 0 || wi >= in.W) continue;
        const size_t src = (((size_t)b * in.H + hi_) * in.W + wi) * in.C + c;
        const uint4 h = *reinterpret_cast<const uint4*>(in.hi + src);
        const __half2* hh = reinterpret_cast<const __half2*>(&h);
        float v[8];
#pragma unroll
        for (int t = 0; t < 4; ++t) { const float2 f = __half22float2(hh[t]); v[2 * t] = f.x; v[2 * t + 1] = f.y; }
        if (in.lo != nullptr) {
          const uint4 l = *reinterpret_cast<const uint4*>(in.lo + src);
          const __half2* ll = reinterpret_cast<const __half2*>(&l);
#pragma unroll
          for (int t = 0; t < 4; ++t) { const float2 f = __half22float2(ll[t]); v[2 * t] += f.x; v[2 * t + 1] += f.y; }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) best[j] = fmaxf(best[j], v[j]);
      }
    }
    uint4 h, l;
    __half2* hh = reinterpret_cast<__half2*>(&h);
    __half2* ll = reinterpret_cast<__half2*>(&l);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const __half2 hv = __floats2half2_rn(best[2 * t], best[2 * t + 1]);
      hh[t] = hv;
      const float2 hf = __half22float2(hv);
      ll[t] = __floats2half2_rn(best[2 * t] - hf.x, best[2 * t + 1] - hf.y);
    }
    *reinterpret_cast<uint4*>(out.hi + m * out.C + c) = h;
    if (out.lo != nullptr) *reinterpret_cast<uint4*>(out.lo + m * out.C + c) = l;
  }
}

// ------------------------------------------------------------------------------------------------
// Depthwise cross-correlation, NHWC split planes (engine-internal form of conv2d_dw_group,
// models/rpn.py:32-38): out[b,i,j,c] = sum_{u,v} x[b,i+u,j+v,c] * k[b,u,v,c].
// Thread = (b, output row i, channel pair); it slides a KHxKW register window along j so every
// input element is fetched KH times (rows) instead of KH*KW times; lanes are consecutive channel
// pairs, so each warp load/store is one contiguous 128-byte line.
// Block = (sample b, chunk of XC_CH channels): the whole HxW input tile of those channels is reconstructed to
// fp32 in shared memory once (each element is read from L2 exactly once), then every thread (channel, output
// row) slides a KHxKW window along the row out of smem.  Lanes are consecutive channels: conflict-free LDS and
// contiguous 64-byte stores per plane.
// Register-blocked variant (same mapping idea as xcorr_bulk_sm100.cu): lane = channel (32 consecutive channels of one
// stream: every shared-memory access of a warp is one conflict-free 128-byte row), and a thread owns a
// (row block x column strip) task of NR x SW outputs: per input row SW+KW-1 loads feed NR..KH*SW*KW FMAs.  The tile
// is reconstructed to fp32 in shared memory once; 2 blocks per SM so one block's load phase overlaps the other's math.
template <int KH, int KW, int NR, int SW, int NTHREADS>
__global__ void __launch_bounds__(NTHREADS, 2) xcorr_nhwc_kernel(Act x, const __half* __restrict__ k_hi,
                                                                  const __half* __restrict__ k_lo, Act out,
                                                                  int band_rows, int c_off, float mul,
                                                                  int* __restrict__ ovf) {
  constexpr int XC_CH = 32;
  extern __shared__ float xs[];                  // [(band rows + KH - 1) * W][32]
  const int b = blockIdx.y;
  const int c0 = blockIdx.x * XC_CH;
  const int y0 = blockIdx.z * band_rows;                             // first output row of this block's band
  const int Hob = min(band_rows, out.H - y0);                        // output rows of the band
  const __half* __restrict__ xh = x.hi;
  const __half* __restrict__ xl = x.lo;
  const int npix = (Hob + KH - 1) * x.W;
  const size_t pix0 = (size_t)b * x.H * x.W + (size_t)y0 * x.W;
  // cooperative load: 8 channels (16 B per plane) per item; LD_U items per thread are fetched before any of them is
  // converted, so each thread keeps 2 * LD_U independent 16-byte loads in flight (the tile comes from L2 / HBM:
  // with one item at a time the load phase was latency-bound and dominated the kernel)
  constexpr int LD_U = 4;
  const int nitems = npix * (XC_CH / 8);
  for (int base = threadIdx.x; base < nitems; base += NTHREADS * LD_U) {
    uint4 hbuf[LD_U], lbuf[LD_U];
#pragma unroll
    for (int t = 0; t < LD_U; ++t) {
      const int idx = base + t * NTHREADS;
      if (idx < nitems) {
        const int pix = idx / (XC_CH / 8);
        const int cc = (idx - pix * (XC_CH / 8)) * 8;
        const size_t src = (pix0 + pix) * x.C + c_off + c0 + cc;   // c_off: this branch's slice of a concatenated search conv
        hbuf[t] = *reinterpret_cast<const uint4*>(xh + src);
        lbuf[t] = xl != nullptr ? *reinterpret_cast<const uint4*>(xl + src) : make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int t = 0; t < LD_U; ++t) {
      const int idx = base + t * NTHREADS;
      if (idx < nitems) {
        const int pix = idx / (XC_CH / 8);
        const int cc = (idx - pix * (XC_CH / 8)) * 8;
        const __half2* hh = reinterpret_cast<const __half2*>(&hbuf[t]);
        const __half2* ll = reinterpret_cast<const __half2*>(&lbuf[t]);
        float v[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 f = __half22float2(hh[q]), g = __half22float2(ll[q]);
          v[2 * q] = f.x + g.x;
          v[2 * q + 1] = f.y + g.y;
        }
        float4* dst = reinterpret_cast<float4*>(xs + (size_t)pix * XC_CH + cc);
        dst[0] = make_float4(v[0], v[1], v[2], v[3]);
        dst[1] = make_float4(v[4], v[5], v[6], v[7]);
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = c0 + lane;
  float kk[KH][KW];
#pragma unroll
  for (int u = 0; u < KH; ++u)
#pragma unroll
    for (int v = 0; v < KW; ++v) kk[u][v] = split_load(k_hi, k_lo, (((size_t)b * KH + u) * KW + v) * out.C + c);
  __syncthreads();
  const int Ho = Hob, Wo = out.W, W = x.W;
  // balanced task grid: row blocks of NR or NR-1 rows (25 -> 7,6,6,6), strips of SW or SW-1 columns; tasks are
  // warp-uniform, and the four (rows, cols) shapes get their own straight-line code (no predicated-off FMAs)
  const int nrb = (Ho + NR - 1) / NR, nst = (Wo + SW - 1) / SW;
  const int r_base = Ho / nrb, r_extra = Ho % nrb, c_base = Wo / nst, c_extra = Wo % nst;   // first *_extra blocks get +1
  __half* __restrict__ oh = out.hi;
  __half* __restrict__ ol = out.lo;
  const size_t pix_stride = out.C;
  for (int task = warp; task < nrb * nst; task += NTHREADS / 32) {
    const int rb = task / nst, stp = task - rb * nst;
    const int r0 = rb * r_base + min(rb, r_extra), q0 = stp * c_base + min(stp, c_extra);
    const int nr = r_base + (rb < r_extra ? 1 : 0), nc = c_base + (stp < c_extra ? 1 : 0);
    const float* row = xs + ((size_t)r0 * W + q0) * XC_CH + lane;
    const size_t obase = (((size_t)b * out.H + y0 + r0) * Wo + q0) * pix_stride + c;
    auto run = [&](auto nr_tag, auto nc_tag) {
      constexpr int NRr = decltype(nr_tag)::value, NCc = decltype(nc_tag)::value;
      float acc[NRr][NCc];
#pragma unroll
      for (int i = 0; i < NRr; ++i)
#pragma unroll
        for (int q = 0; q < NCc; ++q) acc[i][q] = 0.f;
#pragma unroll
      for (int r = 0; r < NRr + KH - 1; ++r) {
        float xr[NCc + KW - 1];
#pragma unroll
        for (int q = 0; q < NCc + KW - 1; ++q) xr[q] = row[(r * W + q) * XC_CH];
#pragma unroll
        for (int u = 0; u < KH; ++u) {
          const int i = r - u;
          if (i >= 0 && i < NRr) {
#pragma unroll
            for (int q = 0; q < NCc; ++q)
#pragma unroll
              for (int v = 0; v < KW; ++v) acc[i][q] = fmaf(xr[q + v], kk[u][v], acc[i][q]);
          }
        }
      }
      float amax = 0.f;
      size_t orow = obase;
#pragma unroll
      for (int i = 0; i < NRr; ++i) {
        size_t o = orow;
#pragma unroll
        for (int q = 0; q < NCc; ++q) {
          const float v = acc[i][q] * mul;          // mul = 2^(s_corr - s_search - s_kernel): static activation scales
          amax = fmaxf(amax, fabsf(v));
          const __half hv = __float2half_rn(v);
          oh[o] = hv;
          if (ol != nullptr) ol[o] = __float2half_rn(v - __half2float(hv));
          o += pix_stride;
        }
        orow += (size_t)Wo * pix_stride;
      }
      flag_if_out_of_range(amax, ovf);
    };
    using IR = std::integral_constant<int, NR>;
    using IR1 = std::integral_constant<int, NR - 1>;
    using IC = std::integral_constant<int, SW>;
    using IC1 = std::integral_constant<int, SW - 1>;
    if (nr == NR && nc == SW) run(IR{}, IC{});
    else if (nr == NR && nc == SW - 1) run(IR{}, IC1{});
    else if (nr == NR - 1 && nc == SW) run(IR1{}, IC{});
    else if (nr == NR - 1 && nc == SW - 1) run(IR1{}, IC1{});
    else {
      // any other block shape (response sizes other than 25 / 41): predicated generic code
      float acc[NR][SW];
#pragma unroll
      for (int i = 0; i < NR; ++i)
#pragma unroll
        for (int q = 0; q < SW; ++q) acc[i][q] = 0.f;
#pragma unroll
      for (int r = 0; r < NR + KH - 1; ++r) {
        if (r < nr + KH - 1) {
          float xr[SW + KW - 1];
#pragma unroll
          for (int q = 0; q < SW + KW - 1; ++q) xr[q] = q < nc + KW - 1 ? row[(r * W + q) * XC_CH] : 0.f;
#pragma unroll
          for (int u = 0; u < KH; ++u) {
            const int i = r - u;
            if (i >= 0 && i < NR && i < nr) {
#pragma unroll
              for (int q = 0; q < SW; ++q)
#pragma unroll
                for (int v = 0; v < KW; ++v) acc[i][q] = fmaf(xr[q + v], kk[u][v], acc[i][q]);
            }
          }
        }
      }
      float amax = 0.f;
#pragma unroll
      for (int i = 0; i < NR; ++i)
        if (i < nr) {
#pragma unroll
          for (int q = 0; q < SW; ++q)
            if (q < nc) {
              const float v = acc[i][q] * mul;
              amax = fmaxf(amax, fabsf(v));
              split_store(oh, ol, obase + ((size_t)i * Wo + q) * pix_stride, v);
            }
        }
      flag_if_out_of_range(amax, ovf);
    }
  }
}

// Standalone operator with the reference's own layout (fp32 NCHW, models/rpn.py:32-38): one warp per
// (b,c) plane.  Lane l owns input column j0+l; the KW-wide window is assembled with warp shuffles, so
// every input element is read from memory exactly once per column pass; KH partial output rows are
// carried in registers and retired as soon as their last input row has been consumed.
template <int KH, int KW, int RB>
__global__ void __launch_bounds__(256) xcorr_nchw_kernel(const float* __restrict__ x, const float* __restrict__ k,
                                                         float* __restrict__ out, int planes, int H, int W) {
  const int plane = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (plane >= planes) return;
  const int lane = threadIdx.x & 31;
  const int Ho = H - KH + 1, Wo = W - KW + 1;
  const float* xp = x + (size_t)plane * H * W;
  const float* kp = k + (size_t)plane * KH * KW;
  float* op = out + (size_t)plane * Ho * Wo;
  float kk[KH][KW];
#pragma unroll
  for (int u = 0; u < KH; ++u)
#pragma unroll
    for (int v = 0; v < KW; ++v) kk[u][v] = __ldg(kp + u * KW + v);
  constexpr int COLS = 32 - KW + 1;   // output columns produced per pass
  for (int j0 = 0; j0 < Wo; j0 += COLS) {
    const int col = j0 + lane;
    const bool in_ok = col < W;
    const bool out_ok = lane < COLS && col < Wo;
    float acc[KH];
#pragma unroll
    for (int u = 0; u < KH; ++u) acc[u] = 0.f;
    // RB rows are fetched per batch before any of them is consumed (memory-level parallelism)
    for (int r0 = 0; r0 < H; r0 += RB) {
      float rowv[RB];
#pragma unroll
      for (int t = 0; t < RB; ++t) rowv[t] = (in_ok && r0 + t < H) ? __ldg(xp + (size_t)(r0 + t) * W + col) : 0.f;
#pragma unroll
      for (int t = 0; t < RB; ++t) {
        const int r = r0 + t;
        if (r < H) {   // warp-uniform
          float xv[KW];
          xv[0] = rowv[t];
#pragma unroll
          for (int v = 1; v < KW; ++v) xv[v] = __shfl_down_sync(0xffffffffu, rowv[t], v);
          // acc[u] holds output row r-u
#pragma unroll
          for (int u = 0; u < KH; ++u)
#pragma unroll
            for (int v = 0; v < KW; ++v) acc[u] = fmaf(xv[v], kk[u][v], acc[u]);
          const int done = r - (KH - 1);
          if (done >= 0 && done < Ho && out_ok) op[(size_t)done * Wo + col] = acc[KH - 1];
#pragma unroll
          for (int u = KH - 1; u > 0; --u) acc[u] = acc[u - 1];
          acc[0] = 0.f;
        }
      }
    }
  }
}

// Generic fallback for other kernel sizes (thread per output element).
__global__ void xcorr_nchw_generic_kernel(const float* __restrict__ x, const float* __restrict__ k,
                                          float* __restrict__ out, int planes, int H, int W, int kh, int kw) {
  const int Ho = H - kh + 1, Wo = W - kw + 1;
  const size_t total = (size_t)planes * Ho * Wo;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int j = idx % Wo, i = (idx / Wo) % Ho;
    const size_t pl = idx / ((size_t)Wo * Ho);
    float acc = 0.f;
    for (int u = 0; u < kh; ++u)
      for (int v = 0; v < kw; ++v) acc = fmaf(x[(pl * H + i + u) * W + j + v], k[(pl * kh + u) * kw + v], acc);
    out[idx] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// ResDownS crop x[:, :, 4:-4, 4:-4] (custom.py:21-24) and the refine-stage windows
// pad(f, P)[scale*dy : scale*dy+size, scale*dx : ...] (custom.py:133-135), zero outside the feature map.
__global__ void crop_kernel(Act in, Act out, const int32_t* __restrict__ pos, int scale, int padv, int fixed_off,
                            int pos_max) {
  const size_t total = out.numel() / 8;   // 8 halfs (16 B) per thread
  const int c8n = out.C / 8;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int c = (idx % c8n) * 8;
    const size_t m = idx / c8n;
    const int xo = m % out.W, yo = (m / out.W) % out.H;
    const int b = m / ((size_t)out.W * out.H);
    int yi, xi;
    if (pos != nullptr) {       // positions are clamped to the response map: a bad (dy,dx) must not read out of bounds
      yi = scale * min(max(pos[2 * b], 0), pos_max) + yo - padv;
      xi = scale * min(max(pos[2 * b + 1], 0), pos_max) + xo - padv;
    } else {
      yi = yo + fixed_off;
      xi = xo + fixed_off;
    }
    uint4 h = make_uint4(0, 0, 0, 0), l = make_uint4(0, 0, 0, 0);
    if (yi >= 0 && yi < in.H && xi >= 0 && xi < in.W) {
      const size_t src = (((size_t)b * in.H + yi) * in.W + xi) * in.C + c;
      h = *reinterpret_cast<const uint4*>(in.hi + src);
      if (in.lo != nullptr) l = *reinterpret_cast<const uint4*>(in.lo + src);
    }
    const size_t dst = m * out.C + c;
    *reinterpret_cast<uint4*>(out.hi + dst) = h;
    if (out.lo != nullptr) *reinterpret_cast<uint4*>(out.lo + dst) = l;
  }
}

// p3 = corr_feature[b, :, dy, dx] (custom.py:144-145) as fp32 [B][C]
__global__ void gather_corr_kernel(Act corr, const int32_t* __restrict__ pos, float* __restrict__ out, float mul) {
  const int b = blockIdx.x;
  const int dy = min(max(pos[2 * b], 0), corr.H - 1), dx = min(max(pos[2 * b + 1], 0), corr.W - 1);
  for (int c = threadIdx.x; c < corr.C; c += blockDim.x)
    out[(size_t)b * corr.C + c] =
        mul * split_load(corr.hi, corr.lo, (((size_t)b * corr.H + dy) * corr.W + dx) * corr.C + c);
}

// mask[b, :, dy, dx] of the raw 63*63-channel mask head output (tools/test.py:259-260, the non-refine branch)
__global__ void gather_mask_col_kernel(const float* __restrict__ mask, const int32_t* __restrict__ pos, int C, int R,
                                       float* __restrict__ out) {
  const int b = blockIdx.x;
  const int dy = min(max(pos[2 * b], 0), R - 1), dx = min(max(pos[2 * b + 1], 0), R - 1);
  const float* src = mask + (size_t)b * C * R * R + (size_t)dy * R + dx;
  for (int c = threadIdx.x; c < C; c += blockDim.x) out[(size_t)b * C + c] = src[(size_t)c * R * R];
}

// ConvTranspose2d(256, 32, 15, 15) on a 1x1 input (custom.py:120,149) == [B x Cin] x [Cin x N] + bias,
// N = 15*15*32 ordered (y, x, co) so the result is NHWC fp32.  A thread walks one weight column — a strided walk through
// 7 MB, one DRAM round trip per element, and ptxas keeps only 3-4 of the unrolled loads in flight — so the kernel lasts
// as long as ONE thread's chain: a block is 64 columns x 4 K-slices (chains of Cin/4), 8 samples per thread, partial sums
// reduced through shared memory in a fixed order.
constexpr int DC_BT = 8;      // samples per block
constexpr int DC_COLS = 64;   // output columns per block
constexpr int DC_KS = 4;      // K slices per block
constexpr int DC_KU = 16;     // unrolled weight loads per slice step
__global__ void __launch_bounds__(DC_COLS * DC_KS) deconv_kernel(const float* __restrict__ p3, const float* __restrict__ w,
                                                                 const float* __restrict__ bias, float* __restrict__ out,
                                                                 int B, int Cin, int N, int cout) {
  extern __shared__ float sp3[];             // [DC_BT][Cin], then red[DC_KS][DC_BT][DC_COLS]
  float* red = sp3 + DC_BT * Cin;
  const int b0 = blockIdx.y * DC_BT;
  for (int i = threadIdx.x; i < DC_BT * Cin; i += blockDim.x) {
    const int bb = b0 + i / Cin;
    sp3[i] = bb < B ? p3[(size_t)bb * Cin + i % Cin] : 0.f;
  }
  __syncthreads();
  const int c = threadIdx.x % DC_COLS, ks = threadIdx.x / DC_COLS;
  const int n = blockIdx.x * DC_COLS + c;
  const int nl = n < N ? n : N - 1;          // columns past the end: load a valid one, never stored
  const int kspan = (Cin + DC_KS - 1) / DC_KS;
  const int k0 = ks * kspan, k1 = min(Cin, k0 + kspan);
  float acc[DC_BT];
#pragma unroll
  for (int t = 0; t < DC_BT; ++t) acc[t] = 0.f;
  int k = k0;
  for (; k + DC_KU <= k1; k += DC_KU) {
    float wv[DC_KU];
#pragma unroll
    for (int u = 0; u < DC_KU; ++u) wv[u] = __ldg(w + (size_t)(k + u) * N + nl);
#pragma unroll
    for (int u = 0; u < DC_KU; ++u)
#pragma unroll
      for (int t = 0; t < DC_BT; ++t) acc[t] = fmaf(sp3[t * Cin + k + u], wv[u], acc[t]);
  }
  for (; k < k1; ++k) {
    const float wv = __ldg(w + (size_t)k * N + nl);
#pragma unroll
    for (int t = 0; t < DC_BT; ++t) acc[t] = fmaf(sp3[t * Cin + k], wv, acc[t]);
  }
#pragma unroll
  for (int t = 0; t < DC_BT; ++t) red[(ks * DC_BT + t) * DC_COLS + c] = acc[t];
  __syncthreads();
  if (n >= N) return;
  const float bv = bias[n % cout];
  // slice ks finishes samples ks*2, ks*2+1 (DC_BT / DC_KS each): sum of the K slices in slice order
#pragma unroll
  for (int j = 0; j < DC_BT / DC_KS; ++j) {
    const int t = ks * (DC_BT / DC_KS) + j;
    float v = 0.f;
#pragma unroll
    for (int q = 0; q < DC_KS; ++q) v += red[(q * DC_BT + t) * DC_COLS + c];
    if (b0 + t < B) out[(size_t)(b0 + t) * N + n] = v + bv;
  }
}

// max |hi| of a split-plane activation (calibration of the static activation scales): float bits are monotone for
// non-negative values, so an integer atomicMax on the bits of |v| works; inf / NaN propagate as large bit patterns.
__global__ void absmax_kernel(const __half* __restrict__ hi, size_t n8, float* __restrict__ slot) {
  float m = 0.f;
  unsigned bad = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 v = reinterpret_cast<const uint4*>(hi)[i];
    const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const float2 f = __half22float2(h[t]);
      if (!(fabsf(f.x) <= 65504.f) || !(fabsf(f.y) <= 65504.f)) bad = 1;
      m = fmaxf(m, fmaxf(fabsf(f.x), fabsf(f.y)));
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (bad) m = INFINITY;
    atomicMax(reinterpret_cast<unsigned int*>(slot), __float_as_uint(m));
  }
}

// NCHW fp32 -> NHWC split planes (standalone-operator entry, sm_conv2d).
__global__ void import_nchw_kernel(const float* __restrict__ x, Act out) {
  const size_t total = out.numel();
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int c = idx % out.C;
    const int w = (idx / out.C) % out.W;
    const int h = (idx / ((size_t)out.C * out.W)) % out.H;
    const int b = idx / ((size_t)out.C * out.W * out.H);
    split_store(out.hi, out.lo, idx, x[(((size_t)b * out.C + c) * out.H + h) * out.W + w]);
  }
}

// NHWC split planes -> NCHW fp32 (exports cached features for parity checks / the Python boundary).
__global__ void export_nchw_kernel(Act in, float* __restrict__ out, float mul) {
  const size_t total = in.numel();
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int w = idx % in.W;
    const int h = (idx / in.W) % in.H;
    const int c = (idx / ((size_t)in.W * in.H)) % in.C;
    const int b = idx / ((size_t)in.W * in.H * in.C);
    out[idx] = mul * split_load(in.hi, in.lo, (((size_t)b * in.H + h) * in.W + w) * in.C + c);
  }
}

// ------------------------------------------------------------------------------------------------
// Refine-stage 3x3 pad-1 convs with 1..32 output channels on fp32 NHWC (custom.py:102-124,150-152).
// The input is up(a (+ b)): an optional second operand (the h_i + v_i sum) and a nearest-neighbour
// upsample (index tables computed on the host exactly as ATen does) are fused into the fetch.
// Thread = one output pixel x CPT output channels; the COUT/CPT threads of a pixel are adjacent lanes
// (their input loads coalesce into one broadcast, their weight reads are consecutive float4s);
// weights [3][3][Cin][COUT] live in smem.
template <int CIN, int COUT, int CPT>
__global__ void __launch_bounds__(256) small_conv3x3_kernel(const float* __restrict__ a, const float* __restrict__ b2,
                                                            int B, int Hi, int Wi, int Ho, int Wo,
                                                            const int* __restrict__ ymap, const int* __restrict__ xmap,
                                                            const float* __restrict__ w, const float* __restrict__ bias,
                                                            int relu, float* __restrict__ out) {
  constexpr int G = COUT / CPT;
  constexpr int NW = 9 * CIN * COUT;
  __shared__ __align__(16) float sw[NW];       // weights [3][3][CIN][COUT], staged once per persistent block
  for (int i = threadIdx.x; i < NW; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const size_t total = (size_t)B * Ho * Wo * G;
  for (size_t gid = blockIdx.x * (size_t)blockDim.x + threadIdx.x; gid < total; gid += (size_t)gridDim.x * blockDim.x) {
    const size_t m = gid / G;
    const int co0 = (int)(gid % G) * CPT;
    const int xo = m % Wo, yo = (m / Wo) % Ho;
    const int b = m / ((size_t)Wo * Ho);
    float acc[CPT];
#pragma unroll
    for (int j = 0; j < CPT; ++j) acc[j] = bias[co0 + j];
#pragma unroll 1
    for (int r = 0; r < 3; ++r) {
      const int y = yo + r - 1;
      if (y < 0 || y >= Ho) continue;
      const int ys = ymap[y];
#pragma unroll 1
      for (int s = 0; s < 3; ++s) {
        const int x = xo + s - 1;
        if (x < 0 || x >= Wo) continue;
        const size_t src = (((size_t)b * Hi + ys) * Wi + xmap[x]) * CIN;
        float vin[CIN];
#pragma unroll
        for (int c = 0; c < CIN; c += 4) {       // all loads of the tap are issued before any math
          const float4 v = *reinterpret_cast<const float4*>(a + src + c);
          vin[c] = v.x; vin[c + 1] = v.y; vin[c + 2] = v.z; vin[c + 3] = v.w;
        }
        if (b2 != nullptr) {
#pragma unroll
          for (int c = 0; c < CIN; c += 4) {
            const float4 v = *reinterpret_cast<const float4*>(b2 + src + c);
            vin[c] += v.x; vin[c + 1] += v.y; vin[c + 2] += v.z; vin[c + 3] += v.w;
          }
        }
        const float* wt = sw + (r * 3 + s) * CIN * COUT + co0;
#pragma unroll
        for (int c = 0; c < CIN; ++c) {
          if constexpr (CPT % 4 == 0) {
#pragma unroll
            for (int j = 0; j < CPT; j += 4) {
              const float4 wv = *reinterpret_cast<const float4*>(wt + c * COUT + j);
              acc[j + 0] = fmaf(vin[c], wv.x, acc[j + 0]);
              acc[j + 1] = fmaf(vin[c], wv.y, acc[j + 1]);
              acc[j + 2] = fmaf(vin[c], wv.z, acc[j + 2]);
              acc[j + 3] = fmaf(vin[c], wv.w, acc[j + 3]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < CPT; ++j) acc[j] = fmaf(vin[c], wt[c * COUT + j], acc[j]);
          }
        }
      }
    }
    float* dst = out + m * COUT + co0;
    if constexpr (CPT % 4 == 0) {
#pragma unroll
      for (int j = 0; j < CPT; j += 4) {
        float4 o = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
        if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        *reinterpret_cast<float4*>(dst + j) = o;
      }
    } else {
#pragma unroll
      for (int j = 0; j < CPT; ++j) dst[j] = relu ? fmaxf(acc[j], 0.f) : acc[j];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Score / box post-processing of siamese_track (tools/test.py:205-254), one block per tracker stream:
//   score = softmax(cls)[:,1]; box = anchor decode of loc (:209-212); scale / ratio penalty (:214-232);
//   pscore = penalty*score*(1-wi) + window*wi (:235-236); argmax (:237, first maximum wins like np.argmax);
//   (dy, dx) = unravel(best, (A, R, R))[1:] (:253-254).
// cls f32 [B][2A][R][R], loc f32 [B][4A][R][R], anchors f32 [A*R*R][4] (cx,cy,w,h), window f32 [A*R*R],
// tsz f64 [B][2] = target_sz * scale_x (float64 as in the reference).  The network part is fp32 as in the reference;
// the penalty is evaluated in fp64 (numpy promotes those expressions to float64 through the float64 target size).
// np.argmax semantics incl. NaN: the first NaN wins over every number (a NaN/Inf network output or a 0/0 target
// size must not leave `besti` unset: rec/pos are always in range).  rec[7] = best index (exact in fp32).
constexpr int SEL_THREADS = 512;   // latency-bound (fp64 exp / divides per candidate): more threads, fewer serial candidates each
__global__ void __launch_bounds__(SEL_THREADS) select_kernel(const float* __restrict__ cls, const float* __restrict__ loc,
                                                     const float* __restrict__ anchors,
                                                     const float* __restrict__ window,
                                                     const double* __restrict__ tsz, int A, int R, double penalty_k,
                                                     double window_influence, int32_t* __restrict__ best_idx,
                                                     int32_t* __restrict__ pos, float* __restrict__ rec) {
  const int b = blockIdx.x;
  const int RR = R * R, n = A * RR;
  const float* c = cls + (size_t)b * 2 * A * RR;
  const float* l = loc + (size_t)b * 4 * A * RR;
  const double tw = tsz[2 * b], th = tsz[2 * b + 1];
  const double tpad = (tw + th) * 0.5;
  const double tsz_c = sqrt((tw + tpad) * (th + tpad));
  const double tratio = tw / th;
  // candidate order: (is NaN, value, -index) — NaN beats every number, ties go to the lower index
  double best = -INFINITY;
  int besti = 0x7fffffff;
  int bestnan = -1;                 // -1: no candidate yet
  auto better = [](int nan_a, double va, int ia, int nan_b, double vb, int ib) {
    if (nan_a != nan_b) return nan_a > nan_b;
    if (nan_a == 1) return ia < ib;
    return va > vb || (va == vb && ia < ib);
  };
  for (int idx = threadIdx.x; idx < n; idx += blockDim.x) {
    const int a = idx / RR, p = idx - a * RR;
    const float s0 = c[(size_t)a * RR + p], s1 = c[(size_t)(A + a) * RR + p];
    const float m = fmaxf(s0, s1);
    const float e0 = expf(s0 - m), e1 = expf(s1 - m);
    const float score = e1 / (e0 + e1);
    const float aw = anchors[4 * idx + 2], ah = anchors[4 * idx + 3];
    const float w = expf(l[(size_t)(2 * A + a) * RR + p]) * aw;
    const float h = expf(l[(size_t)(3 * A + a) * RR + p]) * ah;
    const float pad = (w + h) * 0.5f;
    const float sz = sqrtf((w + pad) * (h + pad));
    double sc = (double)sz / tsz_c;
    sc = fmax(sc, 1.0 / sc);
    double rc = tratio / (double)(w / h);
    rc = fmax(rc, 1.0 / rc);
    const double penalty = exp(-(rc * sc - 1.0) * penalty_k);
    const double ps = penalty * (double)score * (1.0 - window_influence) + (double)window[idx] * window_influence;
    const int isn = ps != ps ? 1 : 0;
    if (better(isn, ps, idx, bestnan, best, besti)) { best = ps; besti = idx; bestnan = isn; }
  }
  __shared__ double sv[SEL_THREADS];
  __shared__ int si[SEL_THREADS];
  __shared__ int sn[SEL_THREADS];
  sv[threadIdx.x] = best;
  si[threadIdx.x] = besti;
  sn[threadIdx.x] = bestnan;
  __syncthreads();
  for (int s = SEL_THREADS / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      if (better(sn[threadIdx.x + s], sv[threadIdx.x + s], si[threadIdx.x + s], sn[threadIdx.x], sv[threadIdx.x],
                 si[threadIdx.x])) {
        sv[threadIdx.x] = sv[threadIdx.x + s]; si[threadIdx.x] = si[threadIdx.x + s]; sn[threadIdx.x] = sn[threadIdx.x + s];
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int idx = min(max(si[0], 0), n - 1);
    const int a = idx / RR, p = idx - a * RR;
    best_idx[b] = idx;
    pos[2 * b] = p / R;          // delta_y
    pos[2 * b + 1] = p % R;      // delta_x
    const float ax = anchors[4 * idx], ay = anchors[4 * idx + 1], aw = anchors[4 * idx + 2], ah = anchors[4 * idx + 3];
    const float s0 = c[(size_t)a * RR + p], s1 = c[(size_t)(A + a) * RR + p];
    const float m = fmaxf(s0, s1);
    const float e0 = expf(s0 - m), e1 = expf(s1 - m);
    const float score = e1 / (e0 + e1);
    const float w = expf(l[(size_t)(2 * A + a) * RR + p]) * aw;
    const float h = expf(l[(size_t)(3 * A + a) * RR + p]) * ah;
    const float pad = (w + h) * 0.5f;
    double sc = (double)sqrtf((w + pad) * (h + pad)) / tsz_c;
    sc = fmax(sc, 1.0 / sc);
    double rc = tratio / (double)(w / h);
    rc = fmax(rc, 1.0 / rc);
    float* o = rec + 8 * b;
    o[0] = l[(size_t)a * RR + p] * aw + ax;
    o[1] = l[(size_t)(A + a) * RR + p] * ah + ay;
    o[2] = w;
    o[3] = h;
    o[4] = score;
    o[5] = (float)exp(-(rc * sc - 1.0) * penalty_k);
    o[6] = (float)sv[0];
    o[7] = (float)idx;
  }
}

// ------------------------------------------------------------------------------------------------
// get_subwindow_tracking on the device (tools/test.py:67-110): crop a sz x sz window whose top-left corner is
// (xmin, ymin) in frame coordinates (may lie outside: those pixels take uint8(avg_chans), :89-100), resize it to
// model x model exactly like cv2.resize(INTER_LINEAR) does for 8-bit images — OpenCV's fixed-point scheme
// (resize.cpp: 11-bit coefficients, HResizeLinear then VResizeLinear:
//  dst = (((b0*(S0>>4))>>16) + ((b1*(S1>>4))>>16) + 2) >> 2; x fractions are clamped at the borders, y ROWS are) —
// and emit the float CHW tensor the network consumes (:61-64).  box = int32 [B][8]: xmin, ymin, sz, avg0, avg1, avg2.
__device__ __forceinline__ void cv_coeff(int d, double scale, int src_n, bool clamp_frac, int& s0, int& a0, int& a1) {
  float f = (float)(((double)d + 0.5) * scale - 0.5);
  int s = (int)floorf(f);
  f -= (float)s;
  if (clamp_frac) {
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= src_n - 1) { f = 0.f; s = src_n - 1; }
  }
  s0 = s;
  a0 = __float2int_rn((1.f - f) * 2048.f);
  a1 = __float2int_rn(f * 2048.f);
}

__global__ void crop_resize_kernel(const uint8_t* __restrict__ frames, size_t frame_stride, int H, int W,
                                   const int32_t* __restrict__ box, int model, float* __restrict__ out) {
  const int b = blockIdx.z;
  const int dx = blockIdx.x * blockDim.x + threadIdx.x;
  const int dy = blockIdx.y * blockDim.y + threadIdx.y;
  if (dx >= model || dy >= model) return;
  const int32_t* bx = box + 8 * b;
  const int xmin = bx[0], ymin = bx[1], sz = bx[2];
  const uint8_t* fr = frames + (size_t)b * frame_stride;
  auto px = [&](int y, int x, int c) -> int {      // pixel of the (virtual, padded) patch
    const int fy = y + ymin, fx = x + xmin;
    if (fy < 0 || fy >= H || fx < 0 || fx >= W) return bx[3 + c];
    return fr[((size_t)fy * W + fx) * 3 + c];
  };
  float* o = out + (size_t)b * 3 * model * model + (size_t)dy * model + dx;
  if (sz == model) {
#pragma unroll
    for (int c = 0; c < 3; ++c) o[(size_t)c * model * model] = (float)px(dy, dx, c);
    return;
  }
  const double scale = 1.0 / ((double)model / (double)sz);
  int sx, ax0, ax1, sy, by0, by1;
  cv_coeff(dx, scale, sz, true, sx, ax0, ax1);
  cv_coeff(dy, scale, sz, false, sy, by0, by1);
  const int x1 = min(sx + 1, sz - 1);
  const int y0 = min(max(sy, 0), sz - 1), y1 = min(max(sy + 1, 0), sz - 1);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int h0 = px(y0, sx, c) * ax0 + px(y0, x1, c) * ax1;
    const int h1 = px(y1, sx, c) * ax0 + px(y1, x1, c) * ax1;
    const int v = (((by0 * (h0 >> 4)) >> 16) + ((by1 * (h1 >> 4)) >> 16) + 2) >> 2;
    o[(size_t)c * model * model] = (float)min(max(v, 0), 255);
  }
}

// ------------------------------------------------------------------------------------------------
// Mask paste-back: crop_back() of siamese_track (tools/test.py:263-282) = cv2.warpAffine(mask f32, M, (W,H),
// INTER_LINEAR, BORDER_CONSTANT, borderValue) restated from OpenCV's imgwarp.cpp: M (forward map, double) is
// inverted in double; source coordinates are generated in fixed point (AB_BITS = 10, 1/32-pixel sub-positions,
// round_delta = 16); the four bilinear weights are float products of the 1-D (1 - f, f) tables; out-of-image taps
// take the border value.  One thread per destination pixel; maps: double [B][6] on the device.
__global__ void warp_affine_kernel(const float* __restrict__ src, int sh, int sw, const double* __restrict__ maps,
                                   float* __restrict__ dst, int dh, int dw, float border) {
  const int b = blockIdx.z;
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= dw || y >= dh) return;
  const double* m = maps + 6 * b;
  double M0 = m[0], M1 = m[1], M2 = m[2], M3 = m[3], M4 = m[4], M5 = m[5];
  double D = M0 * M4 - M1 * M3;
  D = D != 0.0 ? 1.0 / D : 0.0;
  const double A11 = M4 * D, A22 = M0 * D;
  M0 = A11; M1 *= -D; M3 *= -D; M4 = A22;
  const double b1 = -M0 * M2 - M1 * M5, b2 = -M3 * M2 - M4 * M5;
  M2 = b1; M5 = b2;
  const long long adelta = llrint(M0 * x * 1024.0), bdelta = llrint(M3 * x * 1024.0);
  const long long X0 = llrint((M1 * y + M2) * 1024.0) + 16, Y0 = llrint((M4 * y + M5) * 1024.0) + 16;
  const long long X = (X0 + adelta) >> 5, Y = (Y0 + bdelta) >> 5;
  long long sx = X >> 5, sy = Y >> 5;
  sx = sx < -32768 ? -32768 : (sx > 32767 ? 32767 : sx);     // saturate_cast<short>
  sy = sy < -32768 ? -32768 : (sy > 32767 ? 32767 : sy);
  const float fx = (float)(X & 31) / 32.f, fy = (float)(Y & 31) / 32.f;
  const float wx0 = 1.f - fx, wy0 = 1.f - fy;
  const float w00 = wy0 * wx0, w01 = wy0 * fx, w10 = fy * wx0, w11 = fy * fx;
  const float* s = src + (size_t)b * sh * sw;
  auto px = [&](long long yy, long long xx) -> float {
    return (yy >= 0 && yy < sh && xx >= 0 && xx < sw) ? s[yy * sw + xx] : border;
  };
  // same evaluation order as remapBilinear (no fused multiply-add)
  float v = __fmul_rn(px(sy, sx), w00);
  v = __fadd_rn(v, __fmul_rn(px(sy, sx + 1), w01));
  v = __fadd_rn(v, __fmul_rn(px(sy + 1, sx), w10));
  v = __fadd_rn(v, __fmul_rn(px(sy + 1, sx + 1), w11));
  dst[((size_t)b * dh + y) * dw + x] = v;
}


// ------------------------------------------------------------------------------------------------
// Device-resident tracker state (tools/test.py:172-200, 239-249, 263-282, 305-315), one thread per stream, float64 like
// the reference's numpy arithmetic.  state f64 [B][4] = target_pos (x, y), target_sz (w, h).
//   prepare: the search window of the next frame -> crop box for crop_resize_kernel, target_sz * scale_x for the
//            selection penalty, and (scale_x, round(s_x), crop_box x0, y0) kept for the update.
//   update : decoded winner box + score -> lr-smoothed state, clamped to the frame (:305-315); also the forward affine
//            map of crop_back (:263-275) that pastes the 127x127 (or 63x63) mask back into the frame.
__device__ __forceinline__ double py_round(double v) { return rint(v); }   // Python round(): half to even

__global__ void tracker_prepare_kernel(int B, const double* __restrict__ state, const int32_t* __restrict__ avg,
                                       TrackerHp hp, int32_t* __restrict__ boxes, double* __restrict__ tsz,
                                       double* __restrict__ aux) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double px = state[4 * b], py = state[4 * b + 1], sw = state[4 * b + 2], sh = state[4 * b + 3];
  const double wc_x = sh + hp.context_amount * (sw + sh);      // :180-181 (names as in the reference)
  const double hc_x = sw + hp.context_amount * (sw + sh);
  double s_x = sqrt(wc_x * hc_x);
  const double scale_x = (double)hp.exemplar_size / s_x;
  const double d_search = (double)(hp.instance_size - hp.exemplar_size) / 2.0;
  const double pad = d_search / scale_x;
  s_x = s_x + 2.0 * pad;
  const double sxr = py_round(s_x);
  const double c = (sxr + 1.0) / 2.0;                          // get_subwindow_tracking :71-76
  int32_t* bx = boxes + 8 * b;
  bx[0] = (int32_t)py_round(px - c);
  bx[1] = (int32_t)py_round(py - c);
  bx[2] = (int32_t)sxr;
  bx[3] = avg[3 * b]; bx[4] = avg[3 * b + 1]; bx[5] = avg[3 * b + 2];
  bx[6] = 0; bx[7] = 0;
  tsz[2 * b] = sw * scale_x;
  tsz[2 * b + 1] = sh * scale_x;
  aux[4 * b] = scale_x;
  aux[4 * b + 1] = sxr;
  aux[4 * b + 2] = px - sxr / 2.0;                             // crop_box[0], [1] (:187)
  aux[4 * b + 3] = py - sxr / 2.0;
}

__global__ void tracker_update_kernel(int B, double* __restrict__ state, const float* __restrict__ rec,
                                      const double* __restrict__ aux, const int32_t* __restrict__ imsize, TrackerHp hp,
                                      int A, int R, double* __restrict__ maps, double* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double px = state[4 * b], py = state[4 * b + 1], sw = state[4 * b + 2], sh = state[4 * b + 3];
  const double scale_x = aux[4 * b], sxr = aux[4 * b + 1], cx0 = aux[4 * b + 2], cy0 = aux[4 * b + 3];
  const float* r = rec + 8 * b;
  const float w = r[2], h = r[3], score = r[4];
  // penalty of the winner in float64 exactly as :214-232 evaluates it (float32 box terms, float64 target terms)
  const double tw = sw * scale_x, th = sh * scale_x;
  const double tpad = (tw + th) * 0.5;
  const double tsz_c = sqrt((tw + tpad) * (th + tpad));
  const float padf = (w + h) * 0.5f;
  double sc = (double)sqrtf((w + padf) * (h + padf)) / tsz_c;
  sc = fmax(sc, 1.0 / sc);
  double rc = (tw / th) / (double)(w / h);
  rc = fmax(rc, 1.0 / rc);
  const double penalty = exp(-(rc * sc - 1.0) * hp.penalty_k);
  const double lr = penalty * (double)score * hp.lr;            // :241
  const double p0 = (double)r[0] / scale_x, p1 = (double)r[1] / scale_x, p2 = (double)w / scale_x, p3 = (double)h / scale_x;
  double res_x = p0 + px, res_y = p1 + py;
  double res_w = sw * (1.0 - lr) + p2 * lr, res_h = sh * (1.0 - lr) + p3 * lr;
  const double im_w = imsize[2 * b], im_h = imsize[2 * b + 1];
  if (maps != nullptr) {
    // crop_back mapping of the refined / head mask into the frame (:263-282)
    const int idx = (int)r[7];
    const int pidx = idx % (R * R);
    const double delta_y = pidx / R, delta_x = pidx % R;
    double s = sxr / (double)hp.instance_size;
    const double sb0 = cx0 + (delta_x - hp.base_size / 2.0) * hp.total_stride * s;
    const double sb1 = cy0 + (delta_y - hp.base_size / 2.0) * hp.total_stride * s;
    const double sb2 = s * hp.exemplar_size;
    s = (double)hp.out_size / sb2;
    const double bb0 = -sb0 * s, bb1 = -sb1 * s, bb2 = im_w * s, bb3 = im_h * s;
    const double a = (im_w - 1.0) / bb2, bq = (im_h - 1.0) / bb3;
    double* m = maps + 6 * b;
    m[0] = a; m[1] = 0.0; m[2] = -a * bb0;
    m[3] = 0.0; m[4] = bq; m[5] = -bq * bb1;
  }
  (void)A;
  res_x = fmax(0.0, fmin(im_w, res_x));                         // :305-308
  res_y = fmax(0.0, fmin(im_h, res_y));
  res_w = fmax(10.0, fmin(im_w, res_w));
  res_h = fmax(10.0, fmin(im_h, res_h));
  state[4 * b] = res_x; state[4 * b + 1] = res_y; state[4 * b + 2] = res_w; state[4 * b + 3] = res_h;
  if (out != nullptr) {
    double* o = out + 8 * b;
    o[0] = res_x; o[1] = res_y; o[2] = res_w; o[3] = res_h; o[4] = (double)score; o[5] = penalty; o[6] = lr; o[7] = (double)r[7];
  }
}

// Tiled variant for the 16/32-channel layers (h2, post0, h1): a persistent block stages the weights once, then
// walks 8x16 output tiles: the (upsampled, summed) input halo of a tile is built in shared memory once, every thread
// computes 2 horizontally adjacent pixels x CPT output channels out of smem.  Rows are padded to CIN+1 floats so
// the 8 pixel pairs of a warp hit distinct banks; the COUT/CPT threads of a pair read the same input (broadcast).
constexpr int SCT_H = 8, SCT_W = 16;
template <int CIN, int COUT, int CPT>
__global__ void __launch_bounds__((SCT_H * SCT_W / 2) * (COUT / CPT))
small_conv3x3_tiled_kernel(const float* __restrict__ a, const float* __restrict__ b2, int B, int Hi, int Wi, int Ho, int Wo,
                           const int* __restrict__ ymap, const int* __restrict__ xmap, const float* __restrict__ w,
                           const float* __restrict__ bias, int relu, float* __restrict__ out) {
  constexpr int G = COUT / CPT;
  constexpr int NT = (SCT_H * SCT_W / 2) * G;
  constexpr int ROW = CIN + 1;                                   // padded pixel pitch (floats)
  constexpr int HALO_H = SCT_H + 2, HALO_W = SCT_W + 2;
  extern __shared__ __align__(16) float smem_sc[];
  float* sw = smem_sc;                                           // [9][CIN][COUT]
  float* sin = smem_sc + 9 * CIN * COUT;                         // [HALO_H][HALO_W][ROW]
  for (int i = threadIdx.x; i < 9 * CIN * COUT; i += NT) sw[i] = w[i];
  const int tiles_x = (Wo + SCT_W - 1) / SCT_W, tiles_y = (Ho + SCT_H - 1) / SCT_H;
  const int num_tiles = B * tiles_y * tiles_x;
  const int g = threadIdx.x % G;
  const int pp = threadIdx.x / G;
  const int py = pp / (SCT_W / 2), px0 = (pp % (SCT_W / 2)) * 2;
  const int co0 = g * CPT;
  for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
    const int tx = tile % tiles_x, ty = (tile / tiles_x) % tiles_y, b = tile / (tiles_x * tiles_y);
    const int y0 = ty * SCT_H - 1, x0 = tx * SCT_W - 1;         // halo origin in output coordinates
    __syncthreads();                                             // previous tile's readers are done (and sw is visible)
    for (int i = threadIdx.x; i < HALO_H * HALO_W * (CIN / 4); i += NT) {
      const int c4 = (i % (CIN / 4)) * 4;
      const int hp = i / (CIN / 4);
      const int hy = hp / HALO_W, hx = hp % HALO_W;
      const int y = y0 + hy, x = x0 + hx;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (y >= 0 && y < Ho && x >= 0 && x < Wo) {
        const size_t src = (((size_t)b * Hi + ymap[y]) * Wi + xmap[x]) * CIN + c4;
        v = *reinterpret_cast<const float4*>(a + src);
        if (b2 != nullptr) {
          const float4 v2 = *reinterpret_cast<const float4*>(b2 + src);
          v.x += v2.x; v.y += v2.y; v.z += v2.z; v.w += v2.w;
        }
      }
      float* d = sin + (size_t)hp * ROW + c4;
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    __syncthreads();
    float acc0[CPT], acc1[CPT];
#pragma unroll
    for (int j = 0; j < CPT; ++j) { acc0[j] = bias[co0 + j]; acc1[j] = acc0[j]; }
#pragma unroll 1
    for (int r = 0; r < 3; ++r) {
#pragma unroll 1
      for (int s = 0; s < 3; ++s) {
        const float* in0 = sin + ((size_t)(py + r) * HALO_W + px0 + s) * ROW;
        const float* in1 = in0 + ROW;
        const float* wt = sw + (r * 3 + s) * CIN * COUT + co0;
#pragma unroll 8
        for (int c = 0; c < CIN; ++c) {
          const float a0 = in0[c], a1 = in1[c];
#pragma unroll
          for (int j = 0; j < CPT; j += 4) {
            const float4 wv = *reinterpret_cast<const float4*>(wt + c * COUT + j);
            acc0[j + 0] = fmaf(a0, wv.x, acc0[j + 0]); acc1[j + 0] = fmaf(a1, wv.x, acc1[j + 0]);
            acc0[j + 1] = fmaf(a0, wv.y, acc0[j + 1]); acc1[j + 1] = fmaf(a1, wv.y, acc1[j + 1]);
            acc0[j + 2] = fmaf(a0, wv.z, acc0[j + 2]); acc1[j + 2] = fmaf(a1, wv.z, acc1[j + 2]);
            acc0[j + 3] = fmaf(a0, wv.w, acc0[j + 3]); acc1[j + 3] = fmaf(a1, wv.w, acc1[j + 3]);
          }
        }
      }
    }
    const int oy = ty * SCT_H + py;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int ox = tx * SCT_W + px0 + k;
      if (oy < Ho && ox < Wo) {
        const float* acc = k == 0 ? acc0 : acc1;
        float* dst = out + (((size_t)b * Ho + oy) * Wo + ox) * COUT + co0;
#pragma unroll
        for (int j = 0; j < CPT; j += 4) {
          float4 o = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
          if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
          *reinterpret_cast<float4*>(dst + j) = o;
        }
      }
    }
  }
}

// SM count of the current device (grids of the grid-stride / persistent kernels are sized from it)
inline int device_sms() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int& c = cached[dev & 63];
  if (c == 0 && cudaDeviceGetAttribute(&c, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) c = 148;
  return c;
}
inline int grid_for(size_t total, int block) {
  size_t g = (total + block - 1) / block;
  const size_t cap = (size_t)device_sms() * 64;
  return (int)(g > cap ? cap : (g == 0 ? 1 : g));
}

}  // namespace

// ================================================================================================
void launch_ref_conv(const Act& in, const ConvGeom& g, const float* w, const Epilogue& ep, cudaStream_t st) {
  const int Ho = g.out_size(in.H), Wo = g.out_size(in.W);
  const size_t total = (size_t)in.B * Ho * Wo * g.Cout;
  ref_conv_kernel<<<grid_for(total, 256), 256, 0, st>>>(in, g, w, ep, Ho, Wo);
  SMK_CUDA(cudaGetLastError());
}

void launch_stem(const float* x, int B, int S, const float* w, const float* alpha, const float* beta, Act out,
                 cudaStream_t st) {
  const int So = (S - 7) / 2 + 1;
  SMK_CHECK(out.H == So && out.W == So && out.C == 64 && out.B == B, "stem output shape");
  dim3 grid((So + ST_TW - 1) / ST_TW, (So + ST_TH - 1) / ST_TH, B);
  stem_kernel<<<grid, 256, 0, st>>>(x, S, So, w, alpha, beta, out);
  SMK_CUDA(cudaGetLastError());
}

void launch_maxpool3s2(const Act& in, Act out, cudaStream_t st) {
  SMK_CHECK(out.H == (in.H + 2 - 3) / 2 + 1 && out.C == in.C && out.B == in.B, "maxpool output shape");
  maxpool_kernel<<<grid_for(out.numel() / 8, 256), 256, 0, st>>>(in, out);
  SMK_CUDA(cudaGetLastError());
}

void launch_xcorr_nhwc(const Act& x, int c_off, const __half* k_hi, const __half* k_lo, int kh, int kw, Act out, float mul,
                       int* ovf, cudaStream_t st) {
  SMK_CHECK(kh == 5 && kw == 5, "engine xcorr is specialised for the 5x5 template kernel");
  SMK_CHECK(out.H == x.H - kh + 1 && out.W == x.W - kw + 1 && c_off % 8 == 0 && c_off + out.C <= x.C && out.C % 32 == 0,
            "xcorr shapes");
  // one block = one stream x 32 channels x a band of output rows, its input rows reconstructed to fp32 in smem:
  // 29x29 @255 is one band (105 KB, 2 blocks per SM); 45x45 @383 takes two bands of 21 / 20 rows (144 KB)
  const int Ho = out.H;
  int bands = 1;
  while ((size_t)((Ho + bands - 1) / bands + kh - 1) * x.W * 32 * sizeof(float) > 160 * 1024) ++bands;
  const int band_rows = (Ho + bands - 1) / bands;
  const size_t smem = (size_t)(band_rows + kh - 1) * x.W * 32 * sizeof(float);
  auto kern = xcorr_nhwc_kernel<5, 5, 7, 5, 320>;
  static unsigned long long attr = 0;
  ensure_dynamic_smem(kern, 160 * 1024, attr);
  kern<<<dim3(out.C / 32, x.B, bands), 320, smem, st>>>(x, k_hi, k_lo, out, band_rows, c_off, mul, ovf);
  SMK_CUDA(cudaGetLastError());
}

void launch_xcorr_nchw_f32(const float* x, const float* k, float* out, int planes, int H, int W, int kh, int kw,
                           cudaStream_t st) {
  SMK_CHECK(H >= kh && W >= kw && planes > 0, "xcorr shapes");
  // bulk-copy pipeline (xcorr_bulk_sm100.cu) for whole tiles of planes; the one-warp-per-plane kernel takes the rest
  const int done = launch_xcorr_bulk_f32(x, k, out, planes, H, W, kh, kw, st);
  if (done >= planes) return;
  x += (size_t)done * H * W;
  k += (size_t)done * kh * kw;
  out += (size_t)done * (H - kh + 1) * (W - kw + 1);
  planes -= done;
  if (kh == 5 && kw == 5) {
    const int warps = 8;
    // whole plane in flight when it has at most 32 rows (29 @255), two batches of 24 otherwise (45 @383)
    if (H <= 32) xcorr_nchw_kernel<5, 5, 32><<<(planes + warps - 1) / warps, warps * 32, 0, st>>>(x, k, out, planes, H, W);
    else xcorr_nchw_kernel<5, 5, 24><<<(planes + warps - 1) / warps, warps * 32, 0, st>>>(x, k, out, planes, H, W);
  } else {
    const size_t total = (size_t)planes * (H - kh + 1) * (W - kw + 1);
    xcorr_nchw_generic_kernel<<<grid_for(total, 256), 256, 0, st>>>(x, k, out, planes, H, W, kh, kw);
  }
  SMK_CUDA(cudaGetLastError());
}

void launch_crop_center(const Act& in, int crop, Act out, cudaStream_t st) {
  SMK_CHECK(out.H == in.H - 2 * crop && out.C == in.C && in.C % 8 == 0, "crop shapes");
  crop_kernel<<<grid_for(out.numel() / 8, 256), 256, 0, st>>>(in, out, nullptr, 0, 0, crop, 0);
  SMK_CUDA(cudaGetLastError());
}

void launch_refine_crop(const Act& in, const int32_t* pos, int pos_max, int scale, int padv, int size, Act out,
                        cudaStream_t st) {
  SMK_CHECK(out.H == size && out.W == size && out.C == in.C && in.C % 8 == 0, "refine crop shapes");
  crop_kernel<<<grid_for(out.numel() / 8, 256), 256, 0, st>>>(in, out, pos, scale, padv, 0, pos_max);
  SMK_CUDA(cudaGetLastError());
}

void launch_gather_corr(const Act& corr, const int32_t* pos, float* out, float mul, cudaStream_t st) {
  gather_corr_kernel<<<corr.B, 256, 0, st>>>(corr, pos, out, mul);
  SMK_CUDA(cudaGetLastError());
}

void launch_gather_mask_col(const float* mask, const int32_t* pos, int B, int C, int R, float* out, cudaStream_t st) {
  gather_mask_col_kernel<<<B, 256, 0, st>>>(mask, pos, C, R, out);
  SMK_CUDA(cudaGetLastError());
}

void launch_deconv(const float* p3, const float* w, const float* bias, float* out, int B, int Cin, int N, int cout,
                   cudaStream_t st) {
  dim3 grid((N + DC_COLS - 1) / DC_COLS, (B + DC_BT - 1) / DC_BT);
  const size_t smem = (size_t)(DC_BT * Cin + DC_KS * DC_BT * DC_COLS) * sizeof(float);
  SMK_CHECK(smem <= 48 * 1024, "deconv: Cin too large for the staged samples");
  deconv_kernel<<<grid, DC_COLS * DC_KS, smem, st>>>(p3, w, bias, out, B, Cin, N, cout);
  SMK_CUDA(cudaGetLastError());
}

void launch_absmax(const Act& a, float* slot, cudaStream_t st) {
  SMK_CHECK(a.numel() % 8 == 0, "absmax: element count");
  absmax_kernel<<<grid_for(a.numel() / 8, 256), 256, 0, st>>>(a.hi, a.numel() / 8, slot);
  SMK_CUDA(cudaGetLastError());
}

void launch_split_to_f32(const Act& in, float* out, cudaStream_t st, float mul) {
  export_nchw_kernel<<<grid_for(in.numel(), 256), 256, 0, st>>>(in, out, mul);
  SMK_CUDA(cudaGetLastError());
}

void launch_import_nchw(const float* x, Act out, cudaStream_t st) {
  import_nchw_kernel<<<grid_for(out.numel(), 256), 256, 0, st>>>(x, out);
  SMK_CUDA(cudaGetLastError());
}

void launch_warp_affine(const float* src, int sh, int sw, const double* maps, float* dst, int dh, int dw, float border,
                        int B, cudaStream_t st) {
  dim3 block(32, 8), grid((dw + 31) / 32, (dh + 7) / 8, B);
  warp_affine_kernel<<<grid, block, 0, st>>>(src, sh, sw, maps, dst, dh, dw, border);
  SMK_CUDA(cudaGetLastError());
}

void launch_select(const float* cls, const float* loc, const float* anchors, const float* window, const double* tsz,
                   int B, int A, int R, double penalty_k, double window_influence, int32_t* best_idx, int32_t* pos,
                   float* rec, cudaStream_t st) {
  select_kernel<<<B, SEL_THREADS, 0, st>>>(cls, loc, anchors, window, tsz, A, R, penalty_k, window_influence, best_idx, pos, rec);
  SMK_CUDA(cudaGetLastError());
}

void launch_tracker_prepare(int B, const double* state, const int32_t* avg, const TrackerHp& hp, int32_t* boxes,
                            double* tsz, double* aux, cudaStream_t st) {
  tracker_prepare_kernel<<<(B + 127) / 128, 128, 0, st>>>(B, state, avg, hp, boxes, tsz, aux);
  SMK_CUDA(cudaGetLastError());
}

void launch_tracker_update(int B, double* state, const float* rec, const double* aux, const int32_t* imsize,
                           const TrackerHp& hp, int A, int R, double* maps, double* out, cudaStream_t st) {
  tracker_update_kernel<<<(B + 127) / 128, 128, 0, st>>>(B, state, rec, aux, imsize, hp, A, R, maps, out);
  SMK_CUDA(cudaGetLastError());
}

void launch_crop_resize(const uint8_t* frames, size_t frame_stride, int H, int W, const int32_t* box, int B, int model,
                        float* out, cudaStream_t st) {
  dim3 block(32, 8), grid((model + 31) / 32, (model + 7) / 8, B);
  crop_resize_kernel<<<grid, block, 0, st>>>(frames, frame_stride, H, W, box, model, out);
  SMK_CUDA(cudaGetLastError());
}

// Host-side nearest-neighbour source index, computed the way ATen does for F.upsample(mode='nearest')
// (custom.py:150-152): src = min(floorf(dst * (float)in / out), in - 1).
std::vector<int> nearest_index_table(int out_size, int in_size) {
  std::vector<int> t(out_size);
  const float scale = (float)in_size / (float)out_size;
  for (int d = 0; d < out_size; ++d) {
    int s = (int)floorf((float)d * scale);
    t[d] = s < in_size - 1 ? s : in_size - 1;
  }
  return t;
}

void launch_small_conv3x3_maps(const float* a, const float* b, int B, int Hi, int Wi, int Ho, int Wo, int Cin, int Cout,
                               const int* ymap, const int* xmap, const float* w, const float* bias, int relu,
                               float* out, cudaStream_t st) {
  const size_t M = (size_t)B * Ho * Wo;
#define SMK_SC(CI, CO, CPT)                                                                                      \
  if (Cin == CI && Cout == CO) {                                                                                 \
    const size_t threads = M * (CO / CPT);                                                                       \
    size_t blocks = (threads + 255) / 256;                                                                       \
    if (blocks > (size_t)device_sms() * 6) blocks = (size_t)device_sms() * 6;                                                                     \
    small_conv3x3_kernel<CI, CO, CPT><<<(unsigned)blocks, 256, 0, st>>>(a, b, B, Hi, Wi, Ho, Wo, ymap, xmap, w,  \
                                                                          bias, relu, out);                      \
    launched = true;                                                                                             \
  }
  bool launched = false;
#define SMK_SCT(CI, CO, CPT)                                                                                     \
  if (Cin == CI && Cout == CO) {                                                                                 \
    constexpr int NT = (SCT_H * SCT_W / 2) * (CO / CPT);                                                         \
    constexpr int SMEM = (9 * CI * CO + (SCT_H + 2) * (SCT_W + 2) * (CI + 1)) * (int)sizeof(float);              \
    static unsigned long long attr = 0;                                                                          \
    ensure_dynamic_smem(small_conv3x3_tiled_kernel<CI, CO, CPT>, SMEM, attr);                                    \
    const int tiles = B * ((Ho + SCT_H - 1) / SCT_H) * ((Wo + SCT_W - 1) / SCT_W);                               \
    const int blocks = tiles < device_sms() * 2 ? tiles : device_sms() * 2;                                                       \
    small_conv3x3_tiled_kernel<CI, CO, CPT><<<blocks, NT, SMEM, st>>>(a, b, B, Hi, Wi, Ho, Wo, ymap, xmap, w,    \
                                                                       bias, relu, out);                         \
    launched = true;                                                                                             \
  }
  SMK_SCT(32, 32, 8) SMK_SCT(32, 16, 4) SMK_SCT(16, 16, 4)
#undef SMK_SCT
  if (!launched) { SMK_SC(16, 4, 4) SMK_SC(4, 4, 4) SMK_SC(4, 1, 1) }
  SMK_CHECK(launched, "small conv: unsupported (Cin, Cout)");
#undef SMK_SC
  SMK_CUDA(cudaGetLastError());
}

}  // namespace smk
