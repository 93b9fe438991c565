// The photometric distortions of the reference's augmentation chains on the device: B ragged uint8 HWC images through a
// per-image list of pointwise pixel operations (ssdk_pixel_op), in place or into a second buffer with the same layout.
// Reference: data_generator/object_detection_2d_photometric_ops.py -- ConvertDataType (:62-86), ConvertColor (:23-60, i.e.
// cv2.cvtColor on uint8), Hue (:110-133), Saturation (:166-189), Brightness (:225-246), Contrast (:281-304) and ChannelSwap
// (:438-455), in the orders SSDPhotometricDistortions (data_augmentation_chain_original_ssd.py:146-206) and the other chains use.
//
// It is a pass over the sources on their own, ahead of ssdk_assemble_images: the reference distorts the image before
// SSDExpand, so canvas backgrounds are never distorted, and the colour round trip is computed once per source pixel rather
// than once per resize tap.
//
// Arithmetic (restated in oracle/photometric.py):
//   float32 ops  NumPy 2's float32 arithmetic, the Python-float parameter rounded to float32 first (NEP 50); Hue's % is NumPy's
//                remainder: fmodf, then + 180 when the sign differs from the divisor's (so a tiny negative gives exactly 180)
//   TO_U8        np.round (half to even) then astype(uint8); the typed-state rules keep every value in 0..255 there
//   RGB2HSV      OpenCV's RGB2HSV_b: integer division tables with hsv_shift = 12, hue range 180
//   HSV2RGB      OpenCV's HSV2RGB_b as its optimised (AVX2) build computes it: float32 with a fused multiply-add in 1 - s*h and
//                1 - s*(1 - h), result * 255 truncated on whole 32-pixel vectors of a row and rounded to nearest even on the last
//                (width mod 32) pixels, which its scalar code converts.  Bit-exact to the default cv2.cvtColor over all
//                181 x 256 x 256 inputs in either part of a row.
// This file is compiled with --fmad=false: only the explicit __fmaf_rn calls fuse.
//
//   photometric_kernel  grid (chunks, B): the image's op list is read once per CTA into shared memory.  Each image is a head of
//                       < 16 pixels up to the first byte that is 16-byte aligned, a body of whole 16-pixel (48-byte) units moved
//                       with 16-byte loads / stores through shared memory, and a tail of < 16 pixels.
#include "common.cuh"
#include <cmath>
#include <vector>

using namespace ssdk;

namespace {

constexpr int kMaxPixelOps = 64;
constexpr int kThreads = 256;
constexpr int kPixPerThread = 16;                       // 48 bytes = 3 x 16 bytes
constexpr int kPixPerCta = kThreads * kPixPerThread;
constexpr int kHsvShift = 12;
constexpr int kCvVecPixels = 32;                        // pixels per vector iteration of OpenCV's AVX2 HSV2RGB_b

struct Op {
  int op;
  int arg;
  float f;         // a0 rounded to float32
};

__device__ __forceinline__ float clip255(float x) { return fminf(fmaxf(x, 0.f), 255.f); }

__device__ __forceinline__ void rgb2hsv(float& x0, float& x1, float& x2, const int* sdiv, const int* hdiv) {
  const int r = (int)x0, g = (int)x1, b = (int)x2;
  const int v = max(max(b, g), r), vmin = min(min(b, g), r);
  const int diff = v - vmin;
  const int s = (diff * sdiv[v] + (1 << (kHsvShift - 1))) >> kHsvShift;
  int h = v == r ? g - b : (v == g ? b - r + 2 * diff : r - g + 4 * diff);
  h = (h * hdiv[diff] + (1 << (kHsvShift - 1))) >> kHsvShift;
  h += h < 0 ? 180 : 0;
  x0 = (float)h; x1 = (float)s; x2 = (float)v;
}

__device__ __forceinline__ float pick(const float* tab, unsigned i) { return i == 0 ? tab[0] : (i == 1 ? tab[1] : (i == 2 ? tab[2] : tab[3])); }

__device__ __forceinline__ float to_u8(float x, bool round) { return fminf(round ? rintf(x) : truncf(x), 255.f); }

// `scalar`: the pixel lies in the last (width mod 32) pixels of its row
__device__ __forceinline__ void hsv2rgb(float& x0, float& x1, float& x2, bool scalar) {
  const float hscale = 6.f / 180.f;
  const float s = __fmul_rn(x1, 1.f / 255.f), v = __fmul_rn(x2, 1.f / 255.f);
  float h = __fmul_rn(x0, hscale);                                            // 0 <= h <= 8.5: fmod(h, 6) is one exact subtraction
  if (h >= 6.f) h = __fsub_rn(h, 6.f);
  int sector = (int)floorf(h);
  h = __fsub_rn(h, (float)sector);
  if ((unsigned)sector >= 6u) { sector = 0; h = 0.f; }
  float tab[4];
  tab[0] = v;
  tab[1] = __fmul_rn(v, __fsub_rn(1.f, s));
  tab[2] = __fmul_rn(v, __fmaf_rn(-s, h, 1.f));
  tab[3] = __fmul_rn(v, __fmaf_rn(-s, __fsub_rn(1.f, h), 1.f));
  // OpenCV's sector_data, (b, g, r) indices into tab per sector: {1,3,0}, {1,0,2}, {3,0,1}, {0,2,1}, {0,1,3}, {2,1,0}
  constexpr unsigned kR = 0x031120u, kG = 0x112003u, kB = 0x200311u;  // 4 bits per sector, sector 0 lowest
  const float r = pick(tab, (kR >> (4 * sector)) & 15u), g = pick(tab, (kG >> (4 * sector)) & 15u), b = pick(tab, (kB >> (4 * sector)) & 15u);
  x0 = to_u8(__fmul_rn(r, 255.f), scalar);
  x1 = to_u8(__fmul_rn(g, 255.f), scalar);
  x2 = to_u8(__fmul_rn(b, 255.f), scalar);
}

__device__ __forceinline__ float sel3(float a, float b, float c, int i) { return i == 0 ? a : (i == 1 ? b : c); }

// One pixel (index px of an image w pixels wide) through the list.  The state (uint8 / float32) is implied by the list, which the
// host validated; uint8 values are held as integral floats.
__device__ __forceinline__ void apply_ops(uint8_t* p, long long px, int w, const Op* ops, int n, const int* sdiv, const int* hdiv) {
  float x0 = p[0], x1 = p[1], x2 = p[2];
  for (int i = 0; i < n; ++i) {
    const Op o = ops[i];
    switch (o.op) {
      case SSDK_PIXOP_TO_U8:
        x0 = (float)__float2int_rn(x0); x1 = (float)__float2int_rn(x1); x2 = (float)__float2int_rn(x2);
        break;
      case SSDK_PIXOP_RGB2HSV: rgb2hsv(x0, x1, x2, sdiv, hdiv); break;
      case SSDK_PIXOP_HSV2RGB: {
        const long long col = px < (1LL << 32) ? (long long)((unsigned)px % (unsigned)w) : px % w;
        hsv2rgb(x0, x1, x2, col >= w / kCvVecPixels * kCvVecPixels);
        break;
      }
      case SSDK_PIXOP_BRIGHTNESS:
        x0 = clip255(__fadd_rn(x0, o.f)); x1 = clip255(__fadd_rn(x1, o.f)); x2 = clip255(__fadd_rn(x2, o.f));
        break;
      case SSDK_PIXOP_CONTRAST:
        x0 = clip255(__fadd_rn(127.5f, __fmul_rn(o.f, __fsub_rn(x0, 127.5f))));
        x1 = clip255(__fadd_rn(127.5f, __fmul_rn(o.f, __fsub_rn(x1, 127.5f))));
        x2 = clip255(__fadd_rn(127.5f, __fmul_rn(o.f, __fsub_rn(x2, 127.5f))));
        break;
      case SSDK_PIXOP_SATURATION: x1 = clip255(__fmul_rn(x1, o.f)); break;
      case SSDK_PIXOP_HUE: {
        // -180 <= t <= 435, so fmod(t, 180) is t, t - 180 or t - 360, each exact (Sterbenz); then NumPy's sign fix-up
        const float t = __fadd_rn(x0, o.f);
        float m = t >= 360.f ? __fsub_rn(t, 360.f) : (t >= 180.f ? __fsub_rn(t, 180.f) : (t > -180.f ? t : 0.f));
        if (m < 0.f) m = __fadd_rn(m, 180.f);
        x0 = m;
        break;
      }
      case SSDK_PIXOP_CHANNEL_SWAP: {
        const float y0 = x0, y1 = x1, y2 = x2;
        x0 = sel3(y0, y1, y2, o.arg & 255); x1 = sel3(y0, y1, y2, (o.arg >> 8) & 255); x2 = sel3(y0, y1, y2, (o.arg >> 16) & 255);
        break;
      }
      default: break;                                                          // TO_FLOAT
    }
  }
  p[0] = (uint8_t)x0; p[1] = (uint8_t)x1; p[2] = (uint8_t)x2;
}

// Pixels [0, head) are before the first 16-byte aligned pixel boundary; the body is whole 16-pixel units after it.
__device__ __forceinline__ void split(uintptr_t src, uintptr_t dst, long long n, long long& head, long long& body) {
  if ((src & 15) != (dst & 15)) { head = n; body = 0; return; }
  head = (long long)(((16 - (src & 15)) * 11) & 15);                         // 3 * head == -src (mod 16); 11 = 3^-1 mod 16
  if (head > n) head = n;
  body = (n - head) / kPixPerThread * kPixPerThread;
}

__global__ void __launch_bounds__(kThreads) photometric_kernel(const uint8_t* src_all, uint8_t* dst_all, const int64_t* src_offsets,
                                                               const int* src_hw, const ssdk_pixel_op* ops_all, int max_ops) {
  __shared__ Op s_ops[kMaxPixelOps];
  __shared__ int s_n;
  __shared__ int s_sdiv[256], s_hdiv[256];
  __shared__ __align__(16) uint8_t s_pix[kPixPerCta * 3];
  const int b = blockIdx.y;
  const int w = src_hw[2 * b + 1];
  const long long n = (long long)src_hw[2 * b] * w;
  const uint8_t* src = src_all + src_offsets[b];
  uint8_t* dst = dst_all + src_offsets[b];
  const int t = threadIdx.x;
  if (t < max_ops) {
    const ssdk_pixel_op o = ops_all[(size_t)b * max_ops + t];
    s_ops[t].op = o.op; s_ops[t].arg = o.arg; s_ops[t].f = __double2float_rn(o.a0);
  }
  if (t == 0) {
    int k = 0;
    while (k < max_ops && ops_all[(size_t)b * max_ops + k].op != SSDK_PIXOP_END) ++k;
    s_n = k;
  }
  s_sdiv[t] = t ? __double2int_rn(__ddiv_rn((double)(255 << kHsvShift), (double)t)) : 0;             // cvRound, like OpenCV's tables
  s_hdiv[t] = t ? __double2int_rn(__ddiv_rn((double)(180 << kHsvShift), __dmul_rn(6.0, (double)t))) : 0;
  __syncthreads();
  const int nops = s_n;

  long long head, body;
  split(reinterpret_cast<uintptr_t>(src), reinterpret_cast<uintptr_t>(dst), n, head, body);
  // head and tail pixels, one per thread over the grid's x dimension
  const long long n_edge = n - body;
  for (long long i = (long long)blockIdx.x * kThreads + t; i < n_edge; i += (long long)gridDim.x * kThreads) {
    const long long px = i < head ? i : head + body + (i - head);
    uint8_t p[3] = {src[px * 3], src[px * 3 + 1], src[px * 3 + 2]};
    apply_ops(p, px, w, s_ops, nops, s_sdiv, s_hdiv);
    dst[px * 3] = p[0]; dst[px * 3 + 1] = p[1]; dst[px * 3 + 2] = p[2];
  }
  // the body: 16-byte loads into shared memory, one pixel per thread at a time, 16-byte stores
  for (long long c0 = (long long)blockIdx.x * kPixPerCta; c0 < body; c0 += (long long)gridDim.x * kPixPerCta) {
    const int npx = (int)min((long long)kPixPerCta, body - c0);
    const int nvec = npx * 3 / 16;
    const uint4* vs = reinterpret_cast<const uint4*>(src + (head + c0) * 3);
    uint4* vd = reinterpret_cast<uint4*>(dst + (head + c0) * 3);
    uint4* sv = reinterpret_cast<uint4*>(s_pix);
    __syncthreads();
    for (int i = t; i < nvec; i += kThreads) sv[i] = vs[i];
    __syncthreads();
    for (int i = t; i < npx; i += kThreads) apply_ops(s_pix + 3 * i, head + c0 + i, w, s_ops, nops, s_sdiv, s_hdiv);
    __syncthreads();
    for (int i = t; i < nvec; i += kThreads) vd[i] = sv[i];
  }
}

}  // namespace

extern "C" int ssdk_photometric(ssdk_ctx* ctx, const uint8_t* src_dev, uint8_t* dst_dev, const int64_t* src_offsets_dev, const int* src_hw_dev,
                                int B, const ssdk_pixel_op* ops_dev, int max_ops, void* stream_) {
  SSDK_REQUIRE(ctx && src_dev && dst_dev && src_offsets_dev && src_hw_dev && B > 0, "ssdk_photometric: bad argument");
  SSDK_REQUIRE(max_ops >= 0 && max_ops <= kMaxPixelOps, "ssdk_photometric: max_ops must be in 0..%d", kMaxPixelOps);
  SSDK_REQUIRE(max_ops == 0 || ops_dev, "ssdk_photometric: ops_dev is NULL");
  SSDK_REQUIRE(B <= 65535, "ssdk_photometric: batch of %d is too large", B);
  cudaStream_t stream = (cudaStream_t)stream_;
  // The op lists and image sizes are validated on the host before anything is launched.
  std::vector<int> hw((size_t)B * 2);
  std::vector<ssdk_pixel_op> ops((size_t)B * max_ops);
  SSDK_CHECK_CUDA(cudaMemcpyAsync(hw.data(), src_hw_dev, hw.size() * sizeof(int), cudaMemcpyDeviceToHost, stream));
  if (max_ops) SSDK_CHECK_CUDA(cudaMemcpyAsync(ops.data(), ops_dev, ops.size() * sizeof(ssdk_pixel_op), cudaMemcpyDeviceToHost, stream));
  SSDK_CHECK_CUDA(cudaStreamSynchronize(stream));
  long long max_px = 0;
  for (int b = 0; b < B; ++b) {
    const int h = hw[2 * b], w = hw[2 * b + 1];
    SSDK_REQUIRE(h > 0 && w > 0, "ssdk_photometric: image %d is empty (%d x %d)", b, h, w);
    max_px = std::max(max_px, (long long)h * w);
    bool u8 = true;
    for (int i = 0; i < max_ops; ++i) {
      const ssdk_pixel_op& o = ops[(size_t)b * max_ops + i];
      if (o.op == SSDK_PIXOP_END) break;
      switch (o.op) {
        case SSDK_PIXOP_TO_FLOAT: u8 = false; break;
        case SSDK_PIXOP_TO_U8: u8 = true; break;
        case SSDK_PIXOP_RGB2HSV:
        case SSDK_PIXOP_HSV2RGB:
          SSDK_REQUIRE(u8, "ssdk_photometric: image %d, op %d: colour conversion of a float32 image (convert it to uint8 first)", b, i);
          break;
        case SSDK_PIXOP_BRIGHTNESS:
        case SSDK_PIXOP_CONTRAST:
        case SSDK_PIXOP_SATURATION:
        case SSDK_PIXOP_HUE:
          SSDK_REQUIRE(!u8, "ssdk_photometric: image %d, op %d: photometric arithmetic on a uint8 image (convert it to float32 first)", b, i);
          SSDK_REQUIRE(!std::isnan(o.a0), "ssdk_photometric: image %d, op %d: the parameter is NaN", b, i);
          SSDK_REQUIRE(o.op != SSDK_PIXOP_HUE || (o.a0 >= -180.0 && o.a0 <= 180.0),
                       "ssdk_photometric: image %d, op %d: `delta` must be in the closed interval `[-180, 180]`.", b, i);
          SSDK_REQUIRE((o.op != SSDK_PIXOP_CONTRAST && o.op != SSDK_PIXOP_SATURATION) || (o.a0 > 0.0 && std::isfinite(o.a0)),
                       "ssdk_photometric: image %d, op %d: It must be `factor > 0`.", b, i);
          break;
        case SSDK_PIXOP_CHANNEL_SWAP:
          SSDK_REQUIRE((o.arg & 255) <= 2 && ((o.arg >> 8) & 255) <= 2 && ((o.arg >> 16) & 255) <= 2 && (o.arg >> 24) == 0,
                       "ssdk_photometric: image %d, op %d: channel order 0x%x has an index outside 0..2", b, i, o.arg);
          break;
        default:
          SSDK_REQUIRE(false, "ssdk_photometric: image %d: unknown operation %d", b, o.op);
      }
    }
    SSDK_REQUIRE(u8, "ssdk_photometric: image %d: the list ends in float32 state (end it with TO_U8)", b);
  }
  const long long chunks = (max_px + kPixPerCta - 1) / kPixPerCta;
  const dim3 grid((unsigned)std::min(chunks, 65535LL), B);
  photometric_kernel<<<grid, kThreads, 0, stream>>>(src_dev, dst_dev, src_offsets_dev, src_hw_dev, ops_dev, max_ops);
  SSDK_COUNT_LAUNCH(ctx);
  SSDK_CHECK_CUDA(cudaGetLastError());
  return SSDK_OK;
}
