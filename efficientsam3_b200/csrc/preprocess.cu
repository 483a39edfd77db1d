// Image preprocessing on the device: decoded images of any size (uint8 or fp32, any element strides) -> antialiased bilinear
// resize (torch's _upsample_bilinear2d_aa, align_corners=False) -> per-channel affine -> zero pad -> fp32 NCHW [B,3,S,S].
// Replaces the loaders' ResizeLongestSide.apply_image_torch + norm + pad (stage1/data/transforms.py:48-54,
// stage1/data/sa1b_dataset.py:163-171, 216-227, coco_dataset.py:146-153) and SAM2Transforms (sam1_utils.py:17-41).
//
// The filter is separable and evaluated in torch's order: the width pass first, into an fp32 intermediate, then the height
// pass, each a sequential fp32 sum over taps in ascending input index.  Tap tables (first index, count, normalised weights
// per output coordinate) are built by one small prologue kernel with torch's mixed float / double index arithmetic.
//
// Main kernel: one CTA per 64 x 16 output tile of one image, all three channels.  It streams the input rows the tile needs
// in chunks of <= 40 rows: the raw bytes of each row span are staged in shared memory with aligned 16-byte loads, the width
// pass writes a shared fp32 [rows][3][64] tile, and the height pass accumulates into registers.  An input span wider than a
// staging slot (large downscale factors) is walked in column chunks, so every scale factor works.  Tiles wholly inside the
// pad region only store zeros.
#include "common.cuh"

namespace es3 {
namespace {

constexpr int PP_TW = 64, PP_TH = 16, PP_RC = 40, PP_SLOT_ROW = 768, PP_THREADS = 256;
constexpr int PP_VEC_ROW = PP_SLOT_ROW / 16;                 // 16-byte vectors staged per input row
constexpr int PP_STAGE_VECS = (PP_RC * PP_VEC_ROW + PP_THREADS - 1) / PP_THREADS, PP_STAGE_BATCH = 4;
static_assert(PP_STAGE_VECS % PP_STAGE_BATCH == 0, "staging batches");
static_assert(PP_TW == 64 && PP_THREADS % PP_TW == 0, "thread -> column mapping assumes 64-wide tiles");

// Fields of one image descriptor (16 x int64); efficientsam3_b200/stage1/transforms.py builds the same layout.
enum {
  PF_PTR, PF_SC, PF_SH, PF_SW, PF_IN_H, PF_IN_W, PF_OUT_H, PF_OUT_W, PF_DTYPE, PF_PLANES, PF_XC, PF_KX, PF_KY, PF_TAPX,
  PF_TAPY, PF_NFIELDS = 16
};

// One tap record per output coordinate: [first input index, tap count (both int bits), K weights].
__global__ void preprocess_taps_kernel(const long long* __restrict__ table, float* __restrict__ taps) {
  const int b = blockIdx.y, axis = blockIdx.z;   // axis 0: width, 1: height
  const long long* d = table + (long long)b * PF_NFIELDS;
  const int in = (int)d[axis ? PF_IN_H : PF_IN_W], out = (int)d[axis ? PF_OUT_H : PF_OUT_W];
  const int K = (int)d[axis ? PF_KY : PF_KX];
  float* rec0 = taps + d[axis ? PF_TAPY : PF_TAPX];
  // area_pixel_compute_scale / _compute_indices_min_size_weights_aa (aten UpSampleKernel.cpp): float scale and weights,
  // double index arithmetic where C++ promotes to double.  Explicit _rn intrinsics: no contraction into FMAs.
  const float scale = __fdiv_rn((float)in, (float)out);
  const float support = scale >= 1.f ? scale : 1.f;
  const float invscale = scale >= 1.f ? (float)__ddiv_rn(1.0, (double)scale) : 1.f;
  for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < out; o += gridDim.x * blockDim.x) {
    float* rec = rec0 + (long long)o * (K + 2);
    const float center = (float)__dmul_rn((double)scale, (double)o + 0.5);
    const long long lo = (long long)__dadd_rn((double)__fsub_rn(center, support), 0.5);
    const long long hi = (long long)__dadd_rn((double)__fadd_rn(center, support), 0.5);
    const int xmin = (int)(lo > 0 ? lo : 0);
    int xsize = (int)((hi < in ? hi : in) - xmin);
    xsize = xsize < 0 ? 0 : (xsize > K ? K : xsize);
    float total = 0.f;
    for (int j = 0; j < xsize; ++j) {
      const float t = __fsub_rn((float)(j + xmin), center);
      float x = fabsf((float)__dmul_rn(__dadd_rn((double)t, 0.5), (double)invscale));
      const float w = x < 1.f ? __fsub_rn(1.f, x) : 0.f;
      rec[2 + j] = w;
      total = __fadd_rn(total, w);
    }
    if (total != 0.f)
      for (int j = 0; j < xsize; ++j) rec[2 + j] = __fdiv_rn(rec[2 + j], total);
    rec[0] = __int_as_float(xmin);
    rec[1] = __int_as_float(xsize);
  }
}

template <int DT>   // 0: uint8, 1: fp32
__device__ __forceinline__ float stage_px(const unsigned char* stage, int off) {
  if constexpr (DT == 0) return (float)stage[off];
  else return *reinterpret_cast<const float*>(stage + off);
}

template <int DT>
__device__ void preprocess_tile(const long long* __restrict__ d, const float* __restrict__ taps, float* acc, int ox0, int oy0,
                                int tx_last, int ty_last, unsigned char* stage, float* hbuf, int (*rowterm)[3]) {
  const int tid = threadIdx.x, ox = tid & (PP_TW - 1), q0 = tid / PP_TW;
  const unsigned char* img = reinterpret_cast<const unsigned char*>(d[PF_PTR]);
  const int es = DT == 0 ? 1 : 4;
  const long long scb = d[PF_SC] * es, shb = d[PF_SH] * es, swb = d[PF_SW] * es;
  const int planes = (int)d[PF_PLANES], XC = (int)d[PF_XC], Kx = (int)d[PF_KX], Ky = (int)d[PF_KY];
  const float* tx = taps + d[PF_TAPX];
  const float* ty = taps + d[PF_TAPY];
  const int slot = PP_SLOT_ROW / planes, slot_vecs = slot / 16;
  auto rec_x = [&](int o) { return tx + (long long)o * (Kx + 2); };
  auto rec_y = [&](int o) { return ty + (long long)o * (Ky + 2); };
  const int X0 = __float_as_int(rec_x(ox0)[0]);
  const int X1 = __float_as_int(rec_x(tx_last)[0]) + __float_as_int(rec_x(tx_last)[1]);
  const int Y0 = __float_as_int(rec_y(oy0)[0]);
  const int Y1 = __float_as_int(rec_y(ty_last)[0]) + __float_as_int(rec_y(ty_last)[1]);
  // this thread's output column (the width pass visits the same column for every row and channel it handles)
  const bool col_ok = ox0 + ox <= tx_last;
  const float* wx = rec_x(col_ok ? ox0 + ox : tx_last);
  const int xm = __float_as_int(wx[0]), xe = xm + __float_as_int(wx[1]);
  wx += 2;
  for (int r0 = Y0; r0 < Y1; r0 += PP_RC) {
    const int nr = min(PP_RC, Y1 - r0);
    for (int xa = X0; xa < X1; xa += XC) {
      const int xb = min(xa + XC, X1);
      __syncthreads();                                   // the previous chunk's readers of stage / hbuf are done
      // smem offset of element (c, row, x = 0) of each staged row
      if (tid < nr * 3) {
        const int i = tid / 3, c = tid % 3, q = planes == 3 ? c : 0;
        const long long lo = (r0 + i) * shb + q * scb + xa * swb;
        const long long al = (long long)((reinterpret_cast<uintptr_t>(img) + lo) & ~(uintptr_t)15) - (long long)reinterpret_cast<uintptr_t>(img);
        rowterm[i][c] = (int)((i * planes + q) * slot - al + (r0 + i) * shb + c * scb);
      }
      // stage the byte span of every (row, plane) with aligned 16-byte loads (an aligned vector holding a byte of the
      // tensor lies inside its allocation)
      for (int u0 = 0; u0 < PP_STAGE_VECS; u0 += PP_STAGE_BATCH) {   // batches of loads in flight, then their stores
        uint4 v[PP_STAGE_BATCH];
        int dst[PP_STAGE_BATCH];
#pragma unroll
        for (int u = 0; u < PP_STAGE_BATCH; ++u) {
          const int idx = tid + (u0 + u) * PP_THREADS;
          dst[u] = -1;
          if (idx < nr * PP_VEC_ROW) {
            const int i = idx / PP_VEC_ROW, w = idx % PP_VEC_ROW, q = w / slot_vecs, k = w % slot_vecs;
            const long long lo = (r0 + i) * shb + (planes == 3 ? q * scb : 0) + xa * swb;
            const long long hi = (r0 + i) * shb + (planes == 3 ? q * scb : 2 * scb) + (xb - 1) * swb + es;
            const uintptr_t al = (reinterpret_cast<uintptr_t>(img) + lo) & ~(uintptr_t)15;
            const uintptr_t src = al + 16 * (uintptr_t)k;
            if (src < reinterpret_cast<uintptr_t>(img) + hi) {
              v[u] = __ldg(reinterpret_cast<const uint4*>(src));
              dst[u] = (i * planes + q) * slot + 16 * k;
            }
          }
        }
#pragma unroll
        for (int u = 0; u < PP_STAGE_BATCH; ++u)
          if (dst[u] >= 0) *reinterpret_cast<uint4*>(stage + dst[u]) = v[u];
      }
      __syncthreads();
      // width pass: hbuf[i][c][ox] continues the tap sum of the previous column chunk
      if (col_ok) {
        const int j0 = max(xm, xa), j1 = min(xe, xb);
        for (int item = tid; item < nr * 3 * PP_TW; item += PP_THREADS) {
          const int ic = item / PP_TW, i = ic / 3, c = ic % 3;
          float h = xa == X0 ? 0.f : hbuf[item];
          const int base = rowterm[i][c];
          for (int j = j0; j < j1; ++j) h = fmaf(__ldg(wx + (j - xm)), stage_px<DT>(stage, base + (int)(j * swb)), h);
          hbuf[item] = h;
        }
      }
    }
    __syncthreads();
    // height pass over the rows of this chunk
    if (col_ok) {
#pragma unroll
      for (int k = 0; k < 3 * PP_TH / (PP_THREADS / PP_TW); ++k) {
        const int p = q0 + (PP_THREADS / PP_TW) * k, oy = p % PP_TH, c = p / PP_TH;
        if (oy0 + oy > ty_last) continue;
        const float* wy = rec_y(oy0 + oy);
        const int ym = __float_as_int(wy[0]), j0 = max(ym, r0), j1 = min(ym + __float_as_int(wy[1]), r0 + nr);
        for (int j = j0; j < j1; ++j) acc[k] = fmaf(__ldg(wy + 2 + (j - ym)), hbuf[((j - r0) * 3 + c) * PP_TW + ox], acc[k]);
      }
    }
  }
}

constexpr int PP_SMEM = PP_RC * PP_SLOT_ROW + PP_RC * 3 * PP_TW * 4 + PP_RC * 3 * 4;   // stage | hbuf | rowterm

// 3 CTAs (60 KB of shared memory each) per SM
__global__ void __launch_bounds__(PP_THREADS, 3) preprocess_kernel(const long long* __restrict__ table, const float* __restrict__ affine,
                                                                   const float* __restrict__ taps, float* __restrict__ out, int S) {
  extern __shared__ __align__(16) unsigned char pp_smem[];
  unsigned char* stage = pp_smem;
  float* hbuf = reinterpret_cast<float*>(pp_smem + PP_RC * PP_SLOT_ROW);
  int(*rowterm)[3] = reinterpret_cast<int(*)[3]>(pp_smem + PP_RC * PP_SLOT_ROW + PP_RC * 3 * PP_TW * 4);
  constexpr int NK = 3 * PP_TH / (PP_THREADS / PP_TW);
  const int b = blockIdx.z, ox0 = blockIdx.x * PP_TW, oy0 = blockIdx.y * PP_TH;
  const long long* d = table + (long long)b * PF_NFIELDS;
  const int out_h = (int)d[PF_OUT_H], out_w = (int)d[PF_OUT_W];
  float acc[NK];
#pragma unroll
  for (int k = 0; k < NK; ++k) acc[k] = 0.f;
  if (oy0 < out_h && ox0 < out_w) {
    const int tx_last = min(ox0 + PP_TW, out_w) - 1, ty_last = min(oy0 + PP_TH, out_h) - 1;
    if (d[PF_DTYPE] == 0) preprocess_tile<0>(d, taps, acc, ox0, oy0, tx_last, ty_last, stage, hbuf, rowterm);
    else preprocess_tile<1>(d, taps, acc, ox0, oy0, tx_last, ty_last, stage, hbuf, rowterm);
  }
  const int ox = ox0 + (threadIdx.x & (PP_TW - 1)), q0 = threadIdx.x / PP_TW;
  if (ox >= S) return;
  const float* ab = affine + 6 * b;
  float* outb = out + (long long)b * 3 * S * S;
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    const int p = q0 + (PP_THREADS / PP_TW) * k, oy = oy0 + p % PP_TH, c = p / PP_TH;
    if (oy >= S) continue;
    const bool valid = oy < out_h && ox < out_w;        // the reference pads after normalising: exact zeros
    outb[((long long)c * S + oy) * S + ox] = valid ? fmaf(acc[k], ab[c], ab[3 + c]) : 0.f;
  }
}

}  // namespace
}  // namespace es3

// table: [B][16] int64 image descriptors (device); affine: [B][6] fp32 (a_c, b_c); taps: workspace of the size the table's
// tap offsets imply; out: [B,3,S,S] fp32.
extern "C" int es3_preprocess_images(const long long* table, const float* affine, float* taps, int B, int S, int max_out,
                                     float* out, void* stream) {
  using namespace es3;
  ES3_REQUIRE(table && affine && taps && out && B > 0 && S > 0 && max_out > 0 && max_out <= S && B <= 65535,
              "es3_preprocess_images: bad arguments (B=%d S=%d max_out=%d)", B, S, max_out);
  cudaStream_t st = (cudaStream_t)stream;
  static bool smem_set = false;     // the attribute is per function; setting it twice is harmless
  if (!smem_set) {
    ES3_CHECK_CUDA(cudaFuncSetAttribute(preprocess_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PP_SMEM));
    smem_set = true;
  }
  preprocess_taps_kernel<<<dim3(ceil_div(max_out, 128), B, 2), 128, 0, st>>>(table, taps);
  ES3_LAUNCH_CHECK("preprocess_taps_kernel");
  preprocess_kernel<<<dim3(ceil_div(S, PP_TW), ceil_div(S, PP_TH), B), PP_THREADS, PP_SMEM, st>>>(table, affine, taps, out, S);
  ES3_LAUNCH_CHECK("preprocess_kernel");
  return 0;
}
