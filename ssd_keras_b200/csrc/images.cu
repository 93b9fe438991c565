// The image half of the reference's geometric augmentation chain on the device: B ragged uint8 HWC source images through the
// same per-image ssdk_box_op lists ssdk_assemble_batch applies to the boxes, into the (B, H, W, 3) batch the model consumes.
// Reference: the pixel part of CropPad.__call__ (data_generator/object_detection_2d_patch_sampling_ops.py:266-313, used by
// SSDExpand / SSDRandomCrop), Flip (object_detection_2d_geometric_ops.py:171-195) and Resize (:61-72), i.e. cv2.resize on
// 3-channel uint8 for the five modes ResizeRandomInterp draws from (data_augmentation_chain_original_ssd.py:258-266).
//
// No intermediate image is formed.  Crop/pad and flips are integer index maps: every output pixel's resize taps are computed
// in the frame of the image that enters the resize, clamped there like OpenCV clamps them, and mapped back through the
// preceding operations in reverse order.  A tap that leaves the input of a crop/pad operation takes that operation's
// background (walking in reverse, the first such operation met is the one whose canvas holds the pixel).
//
// The interpolation arithmetic is OpenCV's for 8-bit images (imgproc/src/resize.cpp), restated in oracle/augment.py:
//   NEAREST   sx = min(floor(dx * (1 / (W / w_in))), w_in - 1)                                          (resizeNN)
//   LINEAR    11-bit fixed-point taps, vertical pass ((b0*(h0>>4))>>16) + ((b1*(h1>>4))>>16) + 2) >> 2 (VResizeLinearVec_32s8u)
//             exact 2:1 in both axes is the 2x2 area average (cv::resize switches to INTER_AREA there)
//   CUBIC     4 taps, A = -0.75; vertical pass in float32 on whole 8-lane vectors of a row (VResizeCubicVec_32s8u), the
//             last (row length mod 8) values in the integer form (sum + 2^21) >> 22
//   AREA      up-scaling: linear taps with area fractions; integer ratios: integer sums (2x2 rounds half up, other ratios
//             round(sum * (1/area)) in float32); otherwise float32 weights from computeResizeAreaTab, accumulated in OpenCV's order
//   LANCZOS4  8 taps, integer vertical pass (sum + 2^21) >> 22
// This file is compiled with --fmad=false: every double / float expression is rounded step by step like the host code.
//
//   image_ops_kernel  grid (row bands, B): the image's op list is read once into shared memory, the band's row taps are
//                     computed once, each thread computes its columns' taps once and the pixels of the band, the band is
//                     staged in shared memory as uint8 and written with 16-byte stores (float32 or uint8).
#include "common.cuh"
#include <cmath>
#include <vector>

using namespace ssdk;

namespace {

constexpr int kMaxImageOps = 256;
constexpr int kBandRows = 4;
constexpr int kCoefBits = 11;
constexpr int kCoefScale = 1 << kCoefBits;
constexpr int kCubicVecLanes = 8;

enum { KIND_COPY = 0, KIND_NEAREST = 1, KIND_FIXED = 2, KIND_AREA_FAST = 3, KIND_AREA = 4 };
enum { INTER_NEAREST = 0, INTER_LINEAR = 1, INTER_CUBIC = 2, INTER_AREA = 3, INTER_LANCZOS4 = 4 };

// One pixel-moving operation before the resize: h / w = size of the image entering it.
struct PixOp {
  int kind;
  int py, px;
  int h, w;
  unsigned bg;      // CROP_PAD background, R | G << 8 | B << 16
};

struct ImageInfo {
  int n;            // pixel-moving operations before the resize
  int in_h, in_w;   // image entering the resize (= final image without a resize)
  int mode;
  int kind;         // KIND_*
  int fx, fy;       // integer ratios (KIND_AREA_FAST)
};

constexpr double kS45 = 0.70710678118654752440084436210485;
__constant__ double kLanczosCS[8][2] = {{1, 0}, {-kS45, -kS45}, {0, 1}, {kS45, -kS45}, {-1, 0}, {kS45, kS45}, {0, -1}, {-kS45, kS45}};

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Pixel (r, c) of the image that enters the resize, as r | g << 8 | b << 16.
__device__ __forceinline__ unsigned fetch(const uint8_t* __restrict__ src, int sw, const PixOp* ops, int n, int r, int c) {
  for (int i = n - 1; i >= 0; --i) {
    const PixOp& o = ops[i];
    if (o.kind == SSDK_BOXOP_FLIP_H) {
      c = o.w - 1 - c;
    } else if (o.kind == SSDK_BOXOP_FLIP_V) {
      r = o.h - 1 - r;
    } else {
      r += o.py; c += o.px;
      if ((unsigned)r >= (unsigned)o.h || (unsigned)c >= (unsigned)o.w) return o.bg;
    }
  }
  const uint8_t* p = src + ((size_t)r * sw + c) * 3;
  return (unsigned)__ldg(p) | ((unsigned)__ldg(p + 1) << 8) | ((unsigned)__ldg(p + 2) << 16);
}

__device__ __forceinline__ int chan(unsigned v, int ch) { return (int)((v >> (8 * ch)) & 255u); }

__device__ __forceinline__ int fixed_coef(float c) {                  // saturate_cast<short>(c * INTER_RESIZE_COEF_SCALE)
  return clampi(__float2int_rn(__fmul_rn(c, (float)kCoefScale)), -32768, 32767);
}

// Taps of one axis for the separable fixed-point modes: first (unclamped) source index and K coefficients.
// `reset`: the horizontal axis of LINEAR / AREA resets out-of-range taps to the border (fx = 0); the vertical axis does not.
template <int K>
__device__ void axis_taps(int d, int n_in, int n_out, int mode, bool reset, int& first, int* coef) {
  const double inv = (double)n_out / (double)n_in;
  const double scale = 1.0 / inv;
  int s;
  float f;
  if (mode == INTER_AREA) {
    s = (int)floor(__dmul_rn((double)d, scale));
    f = (float)__dsub_rn((double)(d + 1), __dmul_rn((double)(s + 1), inv));
    f = f <= 0.f ? 0.f : __fsub_rn(f, floorf(f));
  } else {
    f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
    s = (int)floorf(f);
    f = __fsub_rn(f, (float)s);
  }
  if (K == 2) {
    if (reset && s < 0) { s = 0; f = 0.f; }
    if (reset && s >= n_in - 1) { s = n_in - 1; f = 0.f; }
    coef[0] = fixed_coef(__fsub_rn(1.f, f));
    coef[1] = kCoefScale - coef[0];
    first = s;
  } else if (K == 4) {                                               // interpolateCubic, A = -0.75
    const float A = -0.75f;
    const float xp1 = __fadd_rn(f, 1.f), omx = __fsub_rn(1.f, f);
    const float c0 = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, xp1), 5.f * A), xp1), 8.f * A), xp1), 4.f * A);
    const float c1 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.f, f), A + 3.f), f), f), 1.f);
    const float c2 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.f, omx), A + 3.f), omx), omx), 1.f);
    const float c3 = __fsub_rn(__fsub_rn(__fsub_rn(1.f, c0), c1), c2);
    coef[0] = fixed_coef(c0); coef[1] = fixed_coef(c1); coef[2] = fixed_coef(c2); coef[3] = fixed_coef(c3);
    first = s - 1;
  } else {                                                           // interpolateLanczos4
    const float x3 = __fadd_rn(f, 3.f);
    const double y0 = __dmul_rn(__dmul_rn(-(double)x3, 3.14159265358979323846), 0.25);
    double s0, c0;
    sincos(y0, &s0, &c0);
    float cb[8], sum = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float y0_ = __fsub_rn(x3, (float)i);
      if (fabsf(y0_) >= 1e-6f) {
        const double y = __dmul_rn(__dmul_rn(-(double)y0_, 3.14159265358979323846), 0.25);
        cb[i] = (float)__ddiv_rn(__dadd_rn(__dmul_rn(kLanczosCS[i][0], s0), __dmul_rn(kLanczosCS[i][1], c0)), __dmul_rn(y, y));
      } else {
        cb[i] = 1e30f;
      }
      sum = __fadd_rn(sum, cb[i]);
    }
    const float rs = __fdiv_rn(1.f, sum);
#pragma unroll
    for (int i = 0; i < 8; ++i) coef[i] = fixed_coef(__fmul_rn(cb[i], rs));
    first = s - 3;
  }
}

// computeResizeAreaTab for one output index: calls fn(source index, float weight) in OpenCV's order.
template <typename Fn>
__device__ __forceinline__ void area_taps(int d, int n_in, int n_out, Fn fn) {
  const double scale = 1.0 / ((double)n_out / (double)n_in);
  const double fs1 = __dmul_rn((double)d, scale);
  const double fs2 = __dadd_rn(fs1, scale);
  const double cell = fmin(scale, __dsub_rn((double)n_in, fs1));
  int s1 = (int)ceil(fs1), s2 = (int)floor(fs2);
  s2 = min(s2, n_in - 1);
  s1 = min(s1, s2);
  if (__dsub_rn((double)s1, fs1) > 1e-3) fn(s1 - 1, (float)__ddiv_rn(__dsub_rn((double)s1, fs1), cell));
  const float full = (float)__ddiv_rn(1.0, cell);
  for (int s = s1; s < s2; ++s) fn(s, full);
  const double tail = __dsub_rn(fs2, (double)s2);
  if (tail > 1e-3) fn(s2, (float)__ddiv_rn(fmin(fmin(tail, 1.0), cell), cell));
}

// Separable fixed-point modes (LINEAR / AREA up-scaling with K = 2, CUBIC with 4, LANCZOS4 with 8): the band's pixels of column x.
template <int K>
__device__ void fixed_column(const uint8_t* __restrict__ src, int sw, const PixOp* ops, const ImageInfo& info, const int* ytap,
                             const int* ybeta, int rows, int x, int out_w, uint8_t* tile) {
  int xfirst, a[K], xs[K];
  axis_taps<K>(x, info.in_w, out_w, info.mode, true, xfirst, a);
#pragma unroll
  for (int t = 0; t < K; ++t) xs[t] = clampi(xfirst + t, 0, info.in_w - 1);
  const int vec_end = out_w * 3 / kCubicVecLanes * kCubicVecLanes;
  for (int r = 0; r < rows; ++r) {
    int h[K][3];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int sy = clampi(ytap[r] + k, 0, info.in_h - 1);
      h[k][0] = h[k][1] = h[k][2] = 0;
#pragma unroll
      for (int t = 0; t < K; ++t) {
        const unsigned v = fetch(src, sw, ops, info.n, sy, xs[t]);
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) h[k][ch] += chan(v, ch) * a[t];
      }
    }
    const int* b = ybeta + r * K;
    uint8_t* o = tile + ((size_t)r * out_w + x) * 3;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      int v;
      if (K == 2) {
        v = (((b[0] * (h[0][ch] >> 4)) >> 16) + ((b[1] * (h[1][ch] >> 4)) >> 16) + 2) >> 2;
      } else if (K == 4 && x * 3 + ch < vec_end) {
        const float scl = 1.f / (float)(kCoefScale * kCoefScale);
        float f = __fmul_rn((float)h[3][ch], __fmul_rn((float)b[3], scl));
        f = __fadd_rn(__fmul_rn((float)h[2][ch], __fmul_rn((float)b[2], scl)), f);
        f = __fadd_rn(__fmul_rn((float)h[1][ch], __fmul_rn((float)b[1], scl)), f);
        f = __fadd_rn(__fmul_rn((float)h[0][ch], __fmul_rn((float)b[0], scl)), f);
        v = __float2int_rn(f);
      } else {
        int s = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) s += b[k] * h[k][ch];
        v = (s + (1 << (2 * kCoefBits - 1))) >> (2 * kCoefBits);
      }
      o[ch] = (uint8_t)clampi(v, 0, 255);
    }
  }
}

__global__ void __launch_bounds__(512) image_ops_kernel(const uint8_t* __restrict__ src_all, const int64_t* __restrict__ src_offsets,
                                                        const int* __restrict__ src_hw, const ssdk_box_op* __restrict__ ops_all,
                                                        int max_ops, int out_h, int out_w, int out_u8, void* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ ImageInfo info;
  __shared__ int s_ytap[kBandRows];
  __shared__ int s_ybeta[kBandRows * 8];
  uint8_t* tile = smem;                                                        // kBandRows * out_w * 3 bytes
  PixOp* s_ops = reinterpret_cast<PixOp*>(smem + ((size_t)kBandRows * out_w * 3 + 15) / 16 * 16);
  const int b = blockIdx.y;
  const int y0 = blockIdx.x * kBandRows;
  const int rows = min(kBandRows, out_h - y0);
  const int sh = src_hw[2 * b], sw = src_hw[2 * b + 1];
  const uint8_t* src = src_all + src_offsets[b];

  if (threadIdx.x == 0) {
    // walk the list: extents, pixel-moving operations before the resize, the resize
    int h = sh, w = sw, n = 0, mode = -1, rh = 0, rw = 0;
    for (int i = 0; i < max_ops; ++i) {
      const ssdk_box_op op = ops_all[(size_t)b * max_ops + i];
      if (op.op == SSDK_BOXOP_END) break;
      if (op.op == SSDK_BOXOP_CROP_PAD || op.op == SSDK_BOXOP_FLIP_H || op.op == SSDK_BOXOP_FLIP_V) {
        PixOp p;
        p.kind = op.op; p.h = h; p.w = w; p.py = 0; p.px = 0; p.bg = 0;
        if (op.op == SSDK_BOXOP_CROP_PAD) {
          p.py = (int)op.a0; p.px = (int)op.a1; p.bg = ((unsigned)op.flags >> 8) & 0xffffffu;
          h = (int)op.a2; w = (int)op.a3;
        }
        s_ops[n++] = p;
      } else if (op.op == SSDK_BOXOP_RESIZE) {
        mode = (op.flags >> 8) & 255; rh = (int)op.a2; rw = (int)op.a3;
      }
    }
    info.n = n; info.in_h = h; info.in_w = w; info.mode = mode; info.fx = info.fy = 1;
    if (mode < 0 || (rh == h && rw == w)) {
      info.kind = KIND_COPY;
    } else if (mode == INTER_NEAREST) {
      info.kind = KIND_NEAREST;
    } else {
      const double sx = 1.0 / ((double)rw / w), sy = 1.0 / ((double)rh / h);
      const int isx = (int)rint(sx), isy = (int)rint(sy);
      const bool fast = fabs(sx - isx) < 2.220446049250313e-16 && fabs(sy - isy) < 2.220446049250313e-16;
      info.fx = isx; info.fy = isy;
      if (mode == INTER_LINEAR && fast && isx == 2 && isy == 2) info.kind = KIND_AREA_FAST;
      else if (mode == INTER_AREA && sx >= 1 && sy >= 1) info.kind = fast ? KIND_AREA_FAST : KIND_AREA;
      else info.kind = KIND_FIXED;
    }
  }
  __syncthreads();
  const int K = info.kind != KIND_FIXED ? 0 : (info.mode == INTER_CUBIC ? 4 : (info.mode == INTER_LANCZOS4 ? 8 : 2));
  if (K && threadIdx.x < rows) {                                               // the band's row taps, once per CTA
    const int r = threadIdx.x;
    int first, beta[8];
    if (K == 2) axis_taps<2>(y0 + r, info.in_h, out_h, info.mode, false, first, beta);
    else if (K == 4) axis_taps<4>(y0 + r, info.in_h, out_h, info.mode, false, first, beta);
    else axis_taps<8>(y0 + r, info.in_h, out_h, info.mode, false, first, beta);
    s_ytap[r] = first;
    for (int k = 0; k < K; ++k) s_ybeta[r * K + k] = beta[k];
  }
  __syncthreads();

  for (int x = threadIdx.x; x < out_w; x += blockDim.x) {
    if (info.kind == KIND_FIXED) {
      if (K == 2) fixed_column<2>(src, sw, s_ops, info, s_ytap, s_ybeta, rows, x, out_w, tile);
      else if (K == 4) fixed_column<4>(src, sw, s_ops, info, s_ytap, s_ybeta, rows, x, out_w, tile);
      else fixed_column<8>(src, sw, s_ops, info, s_ytap, s_ybeta, rows, x, out_w, tile);
      continue;
    }
    for (int r = 0; r < rows; ++r) {
      const int y = y0 + r;
      int v[3];
      if (info.kind == KIND_COPY || info.kind == KIND_NEAREST) {
        int sy = y, sx = x;
        if (info.kind == KIND_NEAREST) {
          sx = min((int)floor(__dmul_rn((double)x, 1.0 / ((double)out_w / info.in_w))), info.in_w - 1);
          sy = min((int)floor(__dmul_rn((double)y, 1.0 / ((double)out_h / info.in_h))), info.in_h - 1);
        }
        const unsigned p = fetch(src, sw, s_ops, info.n, sy, sx);
        v[0] = chan(p, 0); v[1] = chan(p, 1); v[2] = chan(p, 2);
      } else if (info.kind == KIND_AREA_FAST) {
        int s[3] = {0, 0, 0};
        for (int j = 0; j < info.fy; ++j)
          for (int i = 0; i < info.fx; ++i) {
            const unsigned p = fetch(src, sw, s_ops, info.n, y * info.fy + j, x * info.fx + i);
            s[0] += chan(p, 0); s[1] += chan(p, 1); s[2] += chan(p, 2);
          }
        const bool two = info.fx == 2 && info.fy == 2;
        const float scl = __fdiv_rn(1.f, (float)(info.fx * info.fy));
        for (int ch = 0; ch < 3; ++ch) v[ch] = two ? (s[ch] + 2) >> 2 : __float2int_rn(__fmul_rn((float)s[ch], scl));
      } else {                                                                 // KIND_AREA
        float acc[3] = {0.f, 0.f, 0.f};
        bool first_row = true;
        area_taps(y, info.in_h, out_h, [&](int sy, float beta) {
          float buf[3] = {0.f, 0.f, 0.f};
          area_taps(x, info.in_w, out_w, [&](int sx, float alpha) {
            const unsigned p = fetch(src, sw, s_ops, info.n, sy, sx);
            for (int ch = 0; ch < 3; ++ch) buf[ch] = __fadd_rn(buf[ch], __fmul_rn((float)chan(p, ch), alpha));
          });
          for (int ch = 0; ch < 3; ++ch) acc[ch] = first_row ? __fmul_rn(beta, buf[ch]) : __fadd_rn(acc[ch], __fmul_rn(buf[ch], beta));
          first_row = false;
        });
        for (int ch = 0; ch < 3; ++ch) v[ch] = __float2int_rn(acc[ch]);
      }
      uint8_t* o = tile + ((size_t)r * out_w + x) * 3;
      for (int ch = 0; ch < 3; ++ch) o[ch] = (uint8_t)clampi(v[ch], 0, 255);
    }
  }
  __syncthreads();

  // the band is contiguous in the output: 16-byte stores where the destination is aligned
  const size_t n = (size_t)rows * out_w * 3;
  const size_t base = ((size_t)b * out_h + y0) * out_w * 3;
  if (out_u8) {
    uint8_t* dst = reinterpret_cast<uint8_t*>(out) + base;
    size_t i0 = 0;
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      const size_t nv = n / 16;
      for (size_t i = threadIdx.x; i < nv; i += blockDim.x) reinterpret_cast<uint4*>(dst)[i] = reinterpret_cast<const uint4*>(tile)[i];
      i0 = nv * 16;
    }
    for (size_t i = i0 + threadIdx.x; i < n; i += blockDim.x) dst[i] = tile[i];
  } else {
    float* dst = reinterpret_cast<float*>(out) + base;
    size_t i0 = 0;
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      const size_t nv = n / 4;
      for (size_t i = threadIdx.x; i < nv; i += blockDim.x) {
        const uchar4 q = reinterpret_cast<const uchar4*>(tile)[i];
        reinterpret_cast<float4*>(dst)[i] = make_float4((float)q.x, (float)q.y, (float)q.z, (float)q.w);
      }
      i0 = nv * 4;
    }
    for (size_t i = i0 + threadIdx.x; i < n; i += blockDim.x) dst[i] = (float)tile[i];
  }
}

bool integral(double v) { return std::floor(v) == v && std::fabs(v) < 1e9; }

}  // namespace

extern "C" int ssdk_assemble_images(ssdk_ctx* ctx, const uint8_t* src_dev, const int64_t* src_offsets_dev, const int* src_hw_dev, int B,
                                    const ssdk_box_op* ops_dev, int max_ops, int out_h, int out_w, int out_dtype, void* out_dev,
                                    void* stream_) {
  SSDK_REQUIRE(ctx && src_dev && src_offsets_dev && src_hw_dev && out_dev && B > 0, "ssdk_assemble_images: bad argument");
  SSDK_REQUIRE(out_h > 0 && out_w > 0, "ssdk_assemble_images: empty output size (%d, %d)", out_h, out_w);
  SSDK_REQUIRE(out_dtype == 0 || out_dtype == 1, "ssdk_assemble_images: out_dtype must be 0 (float32) or 1 (uint8)");
  SSDK_REQUIRE(max_ops >= 0 && max_ops <= kMaxImageOps, "ssdk_assemble_images: max_ops must be in 0..%d", kMaxImageOps);
  SSDK_REQUIRE(max_ops == 0 || ops_dev, "ssdk_assemble_images: ops_dev is NULL");
  cudaStream_t stream = (cudaStream_t)stream_;
  // The op lists and source sizes are validated on the host before anything is launched.
  std::vector<int> hw((size_t)B * 2);
  std::vector<ssdk_box_op> ops((size_t)B * max_ops);
  SSDK_CHECK_CUDA(cudaMemcpyAsync(hw.data(), src_hw_dev, hw.size() * sizeof(int), cudaMemcpyDeviceToHost, stream));
  if (max_ops) SSDK_CHECK_CUDA(cudaMemcpyAsync(ops.data(), ops_dev, ops.size() * sizeof(ssdk_box_op), cudaMemcpyDeviceToHost, stream));
  SSDK_CHECK_CUDA(cudaStreamSynchronize(stream));
  for (int b = 0; b < B; ++b) {
    int h = hw[2 * b], w = hw[2 * b + 1];
    SSDK_REQUIRE(h > 0 && w > 0, "ssdk_assemble_images: image %d is empty (%d x %d)", b, h, w);
    bool resized = false;
    for (int i = 0; i < max_ops; ++i) {
      const ssdk_box_op& op = ops[(size_t)b * max_ops + i];
      if (op.op == SSDK_BOXOP_END) break;
      if (op.op == SSDK_BOXOP_CROP_PAD) {
        SSDK_REQUIRE(!resized, "ssdk_assemble_images: image %d: crop/pad after the resize", b);
        SSDK_REQUIRE(integral(op.a0) && integral(op.a1) && integral(op.a2) && integral(op.a3),
                     "ssdk_assemble_images: image %d: crop/pad parameters must be integers", b);
        SSDK_REQUIRE(op.a0 <= h && op.a1 <= w, "ssdk_assemble_images: image %d: the patch at (%g, %g) doesn't overlap with the %d x %d image",
                     b, op.a0, op.a1, h, w);
        SSDK_REQUIRE(op.a2 > 0 && op.a3 > 0, "ssdk_assemble_images: image %d: empty patch", b);
        h = (int)op.a2; w = (int)op.a3;
      } else if (op.op == SSDK_BOXOP_FLIP_H || op.op == SSDK_BOXOP_FLIP_V) {
        SSDK_REQUIRE(!resized, "ssdk_assemble_images: image %d: flip after the resize", b);
        SSDK_REQUIRE(op.a0 == (op.op == SSDK_BOXOP_FLIP_H ? w : h), "ssdk_assemble_images: image %d: flip size %g is not the image's (%d x %d)",
                     b, op.a0, h, w);
      } else if (op.op == SSDK_BOXOP_RESIZE) {
        SSDK_REQUIRE(!resized, "ssdk_assemble_images: image %d: more than one resize", b);
        const int mode = (op.flags >> 8) & 255;
        SSDK_REQUIRE(mode <= INTER_LANCZOS4, "ssdk_assemble_images: image %d: interpolation mode %d is not one of 0..4", b, mode);
        SSDK_REQUIRE(op.a0 == h && op.a1 == w, "ssdk_assemble_images: image %d: resize input %g x %g is not the image's %d x %d", b, op.a0,
                     op.a1, h, w);
        SSDK_REQUIRE(integral(op.a2) && integral(op.a3) && op.a2 > 0 && op.a3 > 0, "ssdk_assemble_images: image %d: bad resize target", b);
        h = (int)op.a2; w = (int)op.a3;
        resized = true;
      } else {
        SSDK_REQUIRE(op.op == SSDK_BOXOP_FILTER, "ssdk_assemble_images: image %d: unknown operation %d", b, op.op);
      }
    }
    SSDK_REQUIRE(h == out_h && w == out_w, "ssdk_assemble_images: image %d ends at %d x %d, the batch is %d x %d", b, h, w, out_h, out_w);
  }
  const size_t tile = ((size_t)kBandRows * out_w * 3 + 15) / 16 * 16;
  const size_t smem = tile + (size_t)max_ops * sizeof(PixOp);
  SSDK_REQUIRE(smem <= 200 * 1024, "ssdk_assemble_images: output width %d is too large", out_w);
  cudaFuncAttributes fa;                                                       // the static shared memory counts towards 48 KB too
  SSDK_CHECK_CUDA(cudaFuncGetAttributes(&fa, image_ops_kernel));
  if (smem + fa.sharedSizeBytes > 48 * 1024)
    SSDK_CHECK_CUDA(cudaFuncSetAttribute(image_ops_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int threads = min(512, max(64, (out_w + 31) / 32 * 32));
  const dim3 grid((out_h + kBandRows - 1) / kBandRows, B);
  SSDK_REQUIRE(grid.y <= 65535, "ssdk_assemble_images: batch of %d is too large", B);
  image_ops_kernel<<<grid, threads, smem, stream>>>(src_dev, src_offsets_dev, src_hw_dev, ops_dev, max_ops, out_h, out_w, out_dtype, out_dev);
  SSDK_COUNT_LAUNCH(ctx);
  SSDK_CHECK_CUDA(cudaGetLastError());
  return SSDK_OK;
}
