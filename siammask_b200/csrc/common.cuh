// Shared types for the SiamMask hot-path kernels (sm_100a).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

namespace smk {

// NHWC activation.  Exact precision mode keeps every activation as two fp16 planes,
// value = hi + lo (22 significant bits); fast mode uses the hi plane only (lo == nullptr).
struct Act {
  __half* hi = nullptr;
  __half* lo = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  int sexp = 0;                     // host-side metadata: stored value = true value * 2^sexp (static activation scale)
  __host__ __device__ size_t numel() const { return (size_t)B * H * W * C; }
  __host__ __device__ int M() const { return B * H * W; }
};

struct ConvGeom {
  int Cin, Cout, KH, KW, stride, pad, dil;
  __host__ __device__ int out_size(int in) const { return (in + 2 * pad - dil * (KH - 1) - 1) / stride + 1; }
};

enum OutMode : int { OUT_NHWC_SPLIT = 0, OUT_NHWC_F32 = 1, OUT_NCHW_F32 = 2 };

// Epilogue common to the tensor-core GEMM conv and the SIMT reference conv:
//   v = acc * alpha[c] + beta[c]  (+ residual[m][c])  (relu)  -> out
struct Epilogue {
  const float* alpha = nullptr;   // [Cout] (folded BN scale / pow2 weight de-scaling)
  const float* beta = nullptr;    // [Cout] (folded BN shift or conv bias)
  const __half* res_hi = nullptr; // residual NHWC [M][Cout], split planes
  const __half* res_lo = nullptr;
  __half* out_hi = nullptr;       // OUT_NHWC_SPLIT
  __half* out_lo = nullptr;
  float* out_f32 = nullptr;       // OUT_NHWC_F32 / OUT_NCHW_F32
  int out_mode = OUT_NHWC_SPLIT;
  int relu = 0;
  int* ovf = nullptr;             // OUT_NHWC_SPLIT: set to 1 when a value leaves fp16's range (|v| > 65504 or NaN)
};

// fp16 split planes hold |v| <= 65504: anything larger (or NaN) raises the engine's overflow flag instead of silently
// becoming inf and poisoning everything downstream (engine.cu: calibrate() picks static power-of-two activation scales)
__device__ __forceinline__ void flag_if_out_of_range(float absmax, int* ovf) {
  if (ovf != nullptr && !(absmax <= 65504.f)) atomicOr(ovf, 1);
}

// One K-segment of the implicit GEMM (see conv_gemm_sm100.cu).
struct GemmSegment {
  CUtensorMap tmA[2];  // hi / lo plane.  kind 0, mode 0: 2D [M][Cin]; mode 1: im2col over NHWC; kind 1: residual [M][Cout]
  int kind;            // 0: convolution segment, 1: identity (residual) segment
  int mode;
  int num_kb, cblks, KW;
  int stride, pad, dil;
  int b_col0;          // first column of this segment inside the packed weight matrix
};

// Parameters of the tcgen05 implicit-GEMM convolution kernel (passed by value, __grid_constant__).
struct GemmParams {
  GemmSegment seg[2];
  int nseg;
  CUtensorMap tmB[2];   // weights: hi / lo, 2D [Cout_pad][w_ld], K-major
  CUtensorMap tmOut[2]; // staged epilogue: output planes [M][Cout], box 32 cols x 32 rows, 64B swizzle
  int M, Cout, Ho, Wo;
  int n_tiles, m_tiles;
  int staged;           // 1: epilogue goes smem -> TMA store (NHWC split outputs)
  int reverse_m;        // 1: walk the M tiles from the last to the first (see Engine::conv_into: L2 reuse)
  Epilogue ep;
};

// A convolution input for the GEMM launcher: activation + geometry + where its weights start in the matrix.
struct GemmInput {
  Act in;
  ConvGeom g;
  int w_col0;
};

// hyper-parameters of the tracker loop (utils/tracker_config.py + config_davis.json), mirrors sm_tracker_hp
struct TrackerHp {
  double context_amount, penalty_k, window_influence, lr;
  int32_t exemplar_size, instance_size, total_stride, base_size, out_size, reserved;
};

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

#define SMK_CUDA(expr)                                                                              \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      throw smk::CudaError(std::string(#expr) + " failed: " + cudaGetErrorString(_e) + " at " +    \
                           __FILE__ + ":" + std::to_string(__LINE__));                              \
  } while (0)

#define SMK_CHECK(cond, msg)                                                                        \
  do {                                                                                              \
    if (!(cond)) throw std::runtime_error(std::string("check failed: ") + #cond + " — " + (msg));   \
  } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: remember, per kernel, on which devices it was
// already raised (one process may drive several GPUs).
template <typename K>
inline void ensure_dynamic_smem(K kernel, int bytes, unsigned long long& done_mask) {
  int dev = 0;
  SMK_CUDA(cudaGetDevice(&dev));
  const unsigned long long bit = 1ull << (dev & 63);
  if (done_mask & bit) return;
  SMK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done_mask |= bit;
}

// ---- launchers (defined in the .cu files) ---------------------------------------------------

// conv_gemm_sm100.cu : tensor-core implicit GEMM. nsplit = 1 (fast) or 2 planes (exact, 3 MMAs).
bool gemm_conv_supported(const ConvGeom& g);
void launch_gemm_conv(const Act& in, const ConvGeom& g, const __half* w_hi, const __half* w_lo, int cout_pad,
                      const Epilogue& ep, int nsplit, int num_sms, cudaStream_t st);
// General form: 1-2 conv segments accumulating into the same output, optional identity (residual) segment whose
// diag(2^e) block starts at weight column res_col0 (< 0: none).  w_ld = row length of the weight matrix.
void launch_gemm_multi(const GemmInput* convs, int nconv, const Act* residual, int res_col0, const __half* w_hi,
                       const __half* w_lo, int cout_pad, int w_ld, const Epilogue& ep, int nsplit, int num_sms,
                       cudaStream_t st, bool reverse_m = false);

CUtensorMap make_map_tiled_nd(const __half* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                              const uint32_t* box, int swizzle_bytes);

// conv3x3_patch_sm100.cu : 3x3 / s1 / p1 / Cin == Cout in {64, 128} on a resident input patch (no im2col traffic)
bool patch_conv_supported(const Act& in, const ConvGeom& g);
void launch_conv3x3_patch(const Act& in, const ConvGeom& g, const __half* w_hi, const __half* w_lo, int w_ld,
                          const Epilogue& ep, int nsplit, int num_sms, cudaStream_t st);

// stem_sm100.cu : 7x7/2 stem on the tensor cores (weights [64][192] K-major, k = (r*7+s)*3+c, pow2-scaled)
void launch_stem_tc(const float* x_nchw, int B, int S, const __half* w_hi, const __half* w_lo, const float* alpha,
                    const float* beta, Act out, int num_sms, cudaStream_t st, int* ovf = nullptr);

// simt_kernels.cu
void launch_ref_conv(const Act& in, const ConvGeom& g, const float* w_krsc_cout, const Epilogue& ep,
                     cudaStream_t st);
void launch_stem(const float* x_nchw, int B, int S, const float* w, const float* alpha, const float* beta, Act out,
                 cudaStream_t st);
void launch_maxpool3s2(const Act& in, Act out, cudaStream_t st);
void launch_xcorr_nhwc(const Act& x, int c_off, const __half* k_hi, const __half* k_lo, int kh, int kw, Act out,
                       float mul, int* ovf, cudaStream_t st);
void launch_absmax(const Act& a, float* slot, cudaStream_t st);
void launch_xcorr_nchw_f32(const float* x, const float* k, float* out, int planes, int H, int W, int kh, int kw,
                           cudaStream_t st);
int launch_xcorr_bulk_f32(const float* x, const float* k, float* out, int planes, int H, int W, int kh, int kw,
                          cudaStream_t st);
void launch_crop_center(const Act& in, int crop, Act out, cudaStream_t st);
void launch_refine_crop(const Act& in, const int32_t* pos, int pos_max, int scale, int padv, int size, Act out,
                        cudaStream_t st);
void launch_gather_corr(const Act& corr, const int32_t* pos, float* out, float mul, cudaStream_t st);
void launch_gather_mask_col(const float* mask, const int32_t* pos, int B, int C, int R, float* out, cudaStream_t st);
void launch_deconv(const float* p3, const float* w, const float* bias, float* out, int B, int Cin, int N,
                   int cout, cudaStream_t st);
void launch_split_to_f32(const Act& in, float* out, cudaStream_t st, float mul = 1.f);
void launch_import_nchw(const float* x_nchw, Act out, cudaStream_t st);
void launch_warp_affine(const float* src, int sh, int sw, const double* maps, float* dst, int dh, int dw, float border,
                        int B, cudaStream_t st);
void launch_tracker_prepare(int B, const double* state, const int32_t* avg, const TrackerHp& hp, int32_t* boxes,
                            double* tsz, double* aux, cudaStream_t st);
void launch_tracker_update(int B, double* state, const float* rec, const double* aux, const int32_t* imsize,
                           const TrackerHp& hp, int A, int R, double* maps, double* out, cudaStream_t st);
void launch_crop_resize(const uint8_t* frames, size_t frame_stride, int H, int W, const int32_t* box, int B, int model,
                        float* out, cudaStream_t st);
void launch_select(const float* cls, const float* loc, const float* anchors, const float* window, const double* tsz,
                   int B, int A, int R, double penalty_k, double window_influence, int32_t* best_idx, int32_t* pos,
                   float* rec, cudaStream_t st);
// small-channel fp32 NHWC 3x3 pad-1 conv: in = up(a (+ b)); ymap/xmap: device nearest-upsample source indices
void launch_small_conv3x3_maps(const float* a, const float* b, int B, int Hi, int Wi, int Ho, int Wo, int Cin, int Cout,
                               const int* ymap, const int* xmap, const float* w, const float* bias, int relu,
                               float* out, cudaStream_t st);
std::vector<int> nearest_index_table(int out_size, int in_size);
int gemm_cout_pad(int cout);

}  // namespace smk
