// altcorr.cu — on-the-fly windowed correlation (no 4D volume).
//
// Reference: altcorr_forward_kernel (src/lib/altcorr_kernel.cu:27-149), called per pyramid
// level by AltCorrBlock.corr_fn (src/modules/corr.py:112-131) with fp32 NHWC feature maps.
//   s(iy,ix) = < fmap1[b,h,w,:], fmap2[b, floor(y)-r+iy, floor(x)-r+ix, :] >   (0 outside)
//   corr[b,n,ox*(2r+1)+oy,h,w] = bilinear blend of s(oy..oy+1, ox..ox+1) with (dy,dx).
//
// v1 mapping (CUDA cores, fp32 like the reference): one warp per source pixel, lane t owns
// taps t and t+32 of the 8x8 window and walks the C channels with 128-bit loads; the source
// feature vector is staged once per pixel in shared memory; a block covers 32 consecutive
// pixels and writes the 49 channels with coalesced 128-byte rows.
#include "common.cuh"
#include "launch.cuh"
#include <cstdlib>

namespace {

constexpr int kPixPerBlock = 32;
constexpr int kWarps = 8;

template <int R>
__global__ void __launch_bounds__(kWarps * 32)
altcorr_kernel(const float* __restrict__ fmap1, const float* __restrict__ fmap2,
               const float* __restrict__ coords, float* __restrict__ corr, int S, int H, int W,
               int H2, int W2, int C) {
  constexpr int RD = 2 * R + 1;
  constexpr int NT = (RD + 1) * (RD + 1);          // 64 taps
  static_assert(NT == 64, "lane mapping assumes r = 3");
  extern __shared__ float smem[];
  float* f1s = smem;                               // [kWarps][C]
  float* taps = f1s + kWarps * C;                  // [kWarps][NT]
  float* stage = taps + kWarps * NT;               // [RD*RD][kPixPerBlock+1]

  const int b = blockIdx.z, s = blockIdx.y;
  const int k0 = blockIdx.x * kPixPerBlock;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int HW = H * W;
  const float* f2b = fmap2 + (size_t)b * H2 * W2 * C;

  for (int pp = warp; pp < kPixPerBlock; pp += kWarps) {
    const int k = k0 + pp;
    if (k >= HW) break;                            // warp-uniform
    const float* f1 = fmap1 + ((size_t)b * HW + k) * C;
    for (int c = lane; c < C; c += 32) f1s[warp * C + c] = f1[c];
    const float2 xy = *reinterpret_cast<const float2*>(coords + (((size_t)b * S + s) * HW + k) * 2);
    const float fx0 = floorf(xy.x), fy0 = floorf(xy.y);
    const float dx = xy.x - fx0, dy = xy.y - fy0;
    __syncwarp();
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int t = lane + 32 * half;
      const int iy = t / (RD + 1), ix = t % (RD + 1);
      const int h2 = (int)fy0 - R + iy, w2 = (int)fx0 - R + ix;
      float acc = 0.f;
      if (h2 >= 0 && h2 < H2 && w2 >= 0 && w2 < W2) {
        const float* f2 = f2b + ((size_t)h2 * W2 + w2) * C;
        if ((C & 3) == 0) {
          const float4* f2v = reinterpret_cast<const float4*>(f2);
          const float4* f1v = reinterpret_cast<const float4*>(f1s + warp * C);
          for (int c = 0; c < C / 4; ++c) {
            const float4 a = f1v[c], q = __ldg(f2v + c);
            acc = fmaf(a.x, q.x, acc); acc = fmaf(a.y, q.y, acc);
            acc = fmaf(a.z, q.z, acc); acc = fmaf(a.w, q.w, acc);
          }
        } else {
          for (int c = 0; c < C; ++c) acc = fmaf(f1s[warp * C + c], __ldg(f2 + c), acc);
        }
      }
      taps[warp * NT + t] = acc;
    }
    __syncwarp();
    const float w_se = (1 - dy) * (1 - dx), w_sw = (1 - dy) * dx;
    const float w_ne = dy * (1 - dx), w_nw = dy * dx;
    for (int o = lane; o < RD * RD; o += 32) {
      const int ox = o / RD, oy = o % RD;          // channel = ox*RD + oy
      const float* tw = taps + warp * NT;
      float v = tw[oy * (RD + 1) + ox] * w_se;
      v += tw[oy * (RD + 1) + ox + 1] * w_sw;
      v += tw[(oy + 1) * (RD + 1) + ox] * w_ne;
      v += tw[(oy + 1) * (RD + 1) + ox + 1] * w_nw;
      stage[o * (kPixPerBlock + 1) + pp] = v;
    }
    __syncwarp();
  }
  __syncthreads();
  const int npx = min(kPixPerBlock, HW - k0);
  float* outp = corr + (((size_t)b * S + s) * RD * RD) * HW + k0;
  for (int idx = threadIdx.x; idx < RD * RD * kPixPerBlock; idx += kWarps * 32) {
    const int c = idx / kPixPerBlock, p = idx % kPixPerBlock;
    if (p < npx) outp[(size_t)c * HW + p] = stage[c * (kPixPerBlock + 1) + p];
  }
}


// ---------------------------------------------------------------------------------------
// AltCorrBlock.__call__ in one launch (src/modules/corr.py:112-145, S == 1): half-precision
// NHWC feature pyramids indexed per edge ON THE DEVICE (no gathered / float-converted copies:
// the reference materialises pyramid[i][:, jj].float() per level per call), all levels in one
// grid, fp32 accumulation of exact fp16 products — the same numbers the reference's fp32 kernel
// produces from the same half-valued inputs, up to summation order.
// ---------------------------------------------------------------------------------------
struct AltPyrArgs {
  const __half* pyr[4];
  int Hl[4], Wl[4];
  float inv_scale[4];
  const float* coords;      // [N, H, W, 2]
  const int64_t* ii; const int64_t* jj;
  float* out;               // [N, L*49, H*W]
  int N, H, W, C, L;
};

template <int R>
__global__ void __launch_bounds__(kWarps * 32)
altcorr_pyramid_kernel(const AltPyrArgs a) {
  constexpr int RD = 2 * R + 1;
  constexpr int NT = (RD + 1) * (RD + 1);
  extern __shared__ float smem[];
  float* f1s = smem;                               // [kWarps][C]
  float* taps = f1s + kWarps * a.C;                // [kWarps][NT]
  float* stage = taps + kWarps * NT;               // [RD*RD][kPixPerBlock+1]
  const int e = blockIdx.y, lvl = blockIdx.z;
  const int k0 = blockIdx.x * kPixPerBlock;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int HW = a.H * a.W, C = a.C;
  const int H2 = a.Hl[lvl], W2 = a.Wl[lvl];
  const __half* f1b = a.pyr[0] + (size_t)a.ii[e] * HW * C;
  const __half* f2b = a.pyr[lvl] + (size_t)a.jj[e] * H2 * W2 * C;
  const float sc = a.inv_scale[lvl];

  for (int pp = warp; pp < kPixPerBlock; pp += kWarps) {
    const int k = k0 + pp;
    if (k >= HW) break;                            // warp-uniform
    const __half2* f1 = reinterpret_cast<const __half2*>(f1b + (size_t)k * C);
    for (int c = lane; c < C / 2; c += 32) {
      const float2 v = __half22float2(f1[c]);
      f1s[warp * C + 2 * c] = v.x; f1s[warp * C + 2 * c + 1] = v.y;
    }
    const float2 xy = *reinterpret_cast<const float2*>(a.coords + ((size_t)e * HW + k) * 2);
    const float cx = xy.x * sc, cy = xy.y * sc;
    const float fx0 = floorf(cx), fy0 = floorf(cy);
    const float dx = cx - fx0, dy = cy - fy0;
    __syncwarp();
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int t = lane + 32 * hh;
      const int iy = t / (RD + 1), ix = t % (RD + 1);
      const int h2 = (int)fy0 - R + iy, w2 = (int)fx0 - R + ix;
      float acc = 0.f;
      if (h2 >= 0 && h2 < H2 && w2 >= 0 && w2 < W2) {
        const uint4* f2v = reinterpret_cast<const uint4*>(f2b + ((size_t)h2 * W2 + w2) * C);
        const float4* f1v = reinterpret_cast<const float4*>(f1s + warp * C);
        for (int c = 0; c < C / 8; ++c) {
          const uint4 q = __ldg(f2v + c);
          const float4 a0 = f1v[2 * c], a1 = f1v[2 * c + 1];
          const float2 q0 = __half22float2(*reinterpret_cast<const __half2*>(&q.x));
          const float2 q1 = __half22float2(*reinterpret_cast<const __half2*>(&q.y));
          const float2 q2 = __half22float2(*reinterpret_cast<const __half2*>(&q.z));
          const float2 q3 = __half22float2(*reinterpret_cast<const __half2*>(&q.w));
          acc = fmaf(a0.x, q0.x, acc); acc = fmaf(a0.y, q0.y, acc);
          acc = fmaf(a0.z, q1.x, acc); acc = fmaf(a0.w, q1.y, acc);
          acc = fmaf(a1.x, q2.x, acc); acc = fmaf(a1.y, q2.y, acc);
          acc = fmaf(a1.z, q3.x, acc); acc = fmaf(a1.w, q3.y, acc);
        }
      }
      taps[warp * NT + t] = acc;
    }
    __syncwarp();
    const float w_se = (1 - dy) * (1 - dx), w_sw = (1 - dy) * dx;
    const float w_ne = dy * (1 - dx), w_nw = dy * dx;
    for (int o = lane; o < RD * RD; o += 32) {
      const int ox = o / RD, oy = o % RD;
      const float* tw = taps + warp * NT;
      float v = tw[oy * (RD + 1) + ox] * w_se;
      v += tw[oy * (RD + 1) + ox + 1] * w_sw;
      v += tw[(oy + 1) * (RD + 1) + ox] * w_ne;
      v += tw[(oy + 1) * (RD + 1) + ox + 1] * w_nw;
      stage[o * (kPixPerBlock + 1) + pp] = v;
    }
    __syncwarp();
  }
  __syncthreads();
  const int npx = min(kPixPerBlock, HW - k0);
  float* outp = a.out + (((size_t)e * a.L + lvl) * RD * RD) * HW + k0;
  for (int idx = threadIdx.x; idx < RD * RD * kPixPerBlock; idx += kWarps * 32) {
    const int c = idx / kPixPerBlock, p = idx % kPixPerBlock;
    if (p < npx) outp[(size_t)c * HW + p] = stage[c * (kPixPerBlock + 1) + p];
  }
}


// ---------------------------------------------------------------------------------------
// Tensor-core AltCorrBlock: a WARP takes 16 consecutive source pixels and multiplies their
// feature vectors (A, 16 x 128, registers) with every target pixel inside the bounding box of
// their 8x8 windows (B, streamed straight from L2 as mma fragments), 8 targets per
// mma.sync.m16n8k16 column tile.  For a smooth flow field the box is ~25 x 10 targets, i.e. ~3x
// redundant MACs on the tensor pipe instead of 64 x 128 scalar FMAs per pixel, and each target
// row is fetched once per 16 pixels instead of once per pixel.  Inputs are half (exact products),
// accumulation is fp32: the same numbers as the fp32 kernel up to summation order.
// The logical K order of the MMA is a fixed permutation of the channels (identical for A and
// B) chosen so that every fragment load is one 128-bit vector.
// ---------------------------------------------------------------------------------------
constexpr int kTcWarps = 4;
constexpr int kTcPix = 16 * kTcWarps;      // 64 source pixels per block

__device__ __forceinline__ void mma16816_f32(float (&c)[4], unsigned a0, unsigned a1, unsigned a2,
                                             unsigned a3, unsigned b0, unsigned b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <int R>
__global__ void __launch_bounds__(kTcWarps * 32)
altcorr_tc_kernel(const AltPyrArgs a) {
  constexpr int RD = 2 * R + 1;
  static_assert(RD == 7, "8x8 tap windows");
  __shared__ float taps[kTcWarps][16 * 64];
  __shared__ float frac[kTcWarps][16][2];
  __shared__ float stage[RD * RD][kTcPix + 1];
  const int e = blockIdx.y, lvl = blockIdx.z;
  const int k0 = blockIdx.x * kTcPix;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const int HW = a.H * a.W;
  const int H2 = a.Hl[lvl], W2 = a.Wl[lvl];
  const __half* f1b = a.pyr[0] + (size_t)a.ii[e] * HW * 128;
  const __half* f2b = a.pyr[lvl] + (size_t)a.jj[e] * H2 * W2 * 128;
  const float sc = a.inv_scale[lvl];
  const int kw = k0 + warp * 16;                   // first pixel of this warp

  // ---- window origin of pixel (lane & 15) ----
  const int pk = kw + (lane & 15);
  const bool pvalid = pk < HW;
  int fxi = 0, fyi = 0;
  {
    float cx = 0.f, cy = 0.f;
    if (pvalid) {
      const float2 xy = *reinterpret_cast<const float2*>(a.coords + ((size_t)e * HW + pk) * 2);
      cx = xy.x * sc; cy = xy.y * sc;
    }
    const float fx0 = floorf(cx), fy0 = floorf(cy);
    fxi = (int)fx0; fyi = (int)fy0;
    if (lane < 16) { frac[warp][lane][0] = cx - fx0; frac[warp][lane][1] = cy - fy0; }
  }
  // bounding box of all taps of the valid pixels, clipped to the target image
  const int big = 1 << 28;
  // clamp far-out windows so the box arithmetic cannot overflow; they contribute nothing anyway
  const int cfx = max(-big, min(big, fxi)), cfy = max(-big, min(big, fyi));
  int bx0 = __reduce_min_sync(0xffffffffu, pvalid ? cfx - R : big);
  int bx1 = __reduce_max_sync(0xffffffffu, pvalid ? cfx + R + 1 : -big);
  int by0 = __reduce_min_sync(0xffffffffu, pvalid ? cfy - R : big);
  int by1 = __reduce_max_sync(0xffffffffu, pvalid ? cfy + R + 1 : -big);
  bx0 = max(bx0, 0); by0 = max(by0, 0); bx1 = min(bx1, W2 - 1); by1 = min(by1, H2 - 1);
  const int bw = bx1 - bx0 + 1, bh = by1 - by0 + 1;
  const int nt = (bw > 0 && bh > 0) ? bw * bh : 0;
  // window origins of the two rows (pixels g and g+8) whose accumulators this lane holds
  const int ox_lo = __shfl_sync(0xffffffffu, fxi, g) - R, oy_lo = __shfl_sync(0xffffffffu, fyi, g) - R;
  const int ox_hi = __shfl_sync(0xffffffffu, fxi, g + 8) - R, oy_hi = __shfl_sync(0xffffffffu, fyi, g + 8) - R;
  const bool v_lo = (kw + g) < HW, v_hi = (kw + g + 8) < HW;

  for (int i = lane; i < 16 * 64; i += 32) taps[warp][i] = 0.f;

  // ---- A fragments: pixels g and g+8, all 128 channels (4 k-pairs x one 128-bit vector each) ----
  uint4 Alo[4], Ahi[4];
#pragma unroll
  for (int kp = 0; kp < 4; ++kp) {
    Alo[kp] = v_lo ? __ldg(reinterpret_cast<const uint4*>(f1b + (size_t)(kw + g) * 128 + kp * 32 + t4 * 8))
                   : make_uint4(0, 0, 0, 0);
    Ahi[kp] = v_hi ? __ldg(reinterpret_cast<const uint4*>(f1b + (size_t)(kw + g + 8) * 128 + kp * 32 + t4 * 8))
                   : make_uint4(0, 0, 0, 0);
  }
  __syncwarp();

  // ---- stream the box, 8 targets per column tile ----
  for (int c0 = 0; c0 < nt; c0 += 8) {
    const int tb = c0 + g;                         // the target whose row this lane loads (B: n = g)
    uint4 Bv[4];
    if (tb < nt) {
      const int ty = by0 + tb / bw, tx = bx0 + tb % bw;
      const uint4* rowp = reinterpret_cast<const uint4*>(f2b + ((size_t)ty * W2 + tx) * 128 + t4 * 8);
#pragma unroll
      for (int kp = 0; kp < 4; ++kp) Bv[kp] = __ldg(rowp + kp * 4);
    } else {
#pragma unroll
      for (int kp = 0; kp < 4; ++kp) Bv[kp] = make_uint4(0, 0, 0, 0);
    }
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int kp = 0; kp < 4; ++kp) {
      // k-step 2kp: halves 0..3 of each vector; k-step 2kp+1: halves 4..7
      mma16816_f32(acc, Alo[kp].x, Ahi[kp].x, Alo[kp].y, Ahi[kp].y, Bv[kp].x, Bv[kp].y);
      mma16816_f32(acc, Alo[kp].z, Ahi[kp].z, Alo[kp].w, Ahi[kp].w, Bv[kp].z, Bv[kp].w);
    }
    // scatter the 16x8 tile into the per-pixel 8x8 tap arrays
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int tc = c0 + 2 * t4 + j;
      if (tc < nt) {
        const int ty = by0 + tc / bw, tx = bx0 + tc % bw;
        int iy = ty - oy_lo, ix = tx - ox_lo;
        if (v_lo && (unsigned)iy < 8u && (unsigned)ix < 8u) taps[warp][g * 64 + iy * 8 + ix] = acc[j];
        iy = ty - oy_hi; ix = tx - ox_hi;
        if (v_hi && (unsigned)iy < 8u && (unsigned)ix < 8u) taps[warp][(g + 8) * 64 + iy * 8 + ix] = acc[2 + j];
      }
    }
  }
  __syncwarp();

  // ---- bilinear blend of the tap arrays (x-offset-major channels) ----
  for (int idx = lane; idx < 16 * RD * RD; idx += 32) {
    const int p = idx / (RD * RD), o = idx % (RD * RD);
    const int ox = o / RD, oy = o % RD;
    const float dx = frac[warp][p][0], dy = frac[warp][p][1];
    const float* tw = taps[warp] + p * 64;
    float v = tw[oy * 8 + ox] * ((1 - dy) * (1 - dx));
    v += tw[oy * 8 + ox + 1] * ((1 - dy) * dx);
    v += tw[(oy + 1) * 8 + ox] * (dy * (1 - dx));
    v += tw[(oy + 1) * 8 + ox + 1] * (dy * dx);
    stage[o][warp * 16 + p] = v;
  }
  __syncthreads();
  const int npx = min(kTcPix, HW - k0);
  float* outp = a.out + (((size_t)e * a.L + lvl) * RD * RD) * HW + k0;
  for (int idx = threadIdx.x; idx < RD * RD * kTcPix; idx += kTcWarps * 32) {
    const int c = idx / kTcPix, p = idx % kTcPix;
    if (p < npx) outp[(size_t)c * HW + p] = stage[c][p];
  }
}

}  // namespace

static GsDeviceOnce g_altcorr_once;
static cudaError_t altcorr_device_init(int) {
  cudaError_t e = cudaFuncSetAttribute(altcorr_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(altcorr_pyramid_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  return e;
}

extern "C" {

int goslam_altcorr_forward(const float* fmap1, const float* fmap2, const float* coords,
                           float* corr, int B, int S, int H, int W, int H2, int W2, int C,
                           int radius, void* stream) {
  if (B < 0 || S <= 0 || H <= 0 || W <= 0 || H2 <= 0 || W2 <= 0 || C <= 0) return GOSLAM_EINVAL;
  if (radius != 3) return GOSLAM_EINVAL;
  if (B == 0) return GOSLAM_OK;
  if (S > 65535 || B > 65535) return GOSLAM_EINVAL;
  const size_t smem = (size_t)(kWarps * C + kWarps * 64 + 49 * (kPixPerBlock + 1)) * sizeof(float);
  if (smem > 200 * 1024) return GOSLAM_EINVAL;
  { const int rc = gs_device_once(g_altcorr_once, altcorr_device_init); if (rc != GOSLAM_OK) return rc; }
  dim3 grid(gs_cdiv(H * W, kPixPerBlock), S, B);
  altcorr_kernel<3><<<grid, kWarps * 32, smem, (cudaStream_t)stream>>>(fmap1, fmap2, coords, corr,
                                                                       S, H, W, H2, W2, C);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_altcorr_pyramid(const void* const* pyramid, int num_levels, const float* coords,
                           const int64_t* ii, const int64_t* jj, float* out, int N, int H, int W,
                           int C, int radius, void* stream) {
  if (N < 0 || H <= 0 || W <= 0 || C <= 0 || (C % 8) != 0 || num_levels < 1 || num_levels > 4)
    return GOSLAM_EINVAL;
  if (radius != 3 || N > 65535) return GOSLAM_EINVAL;
  if (N == 0) return GOSLAM_OK;
  AltPyrArgs a{};
  for (int l = 0; l < num_levels; ++l) {
    a.pyr[l] = reinterpret_cast<const __half*>(pyramid[l]);
    a.Hl[l] = H >> l; a.Wl[l] = W >> l;
    a.inv_scale[l] = 1.0f / (float)(1 << l);
    if (a.Hl[l] <= 0 || a.Wl[l] <= 0) return GOSLAM_EINVAL;
  }
  a.coords = coords; a.ii = ii; a.jj = jj; a.out = out;
  a.N = N; a.H = H; a.W = W; a.C = C; a.L = num_levels;
  const size_t smem = (size_t)(kWarps * C + kWarps * 64 + 49 * (kPixPerBlock + 1)) * sizeof(float);
  if (smem > 200 * 1024) return GOSLAM_EINVAL;
  { const int rc = gs_device_once(g_altcorr_once, altcorr_device_init); if (rc != GOSLAM_OK) return rc; }
  if (C == 128) {                   // tensor-core path (the model's feature width)
    dim3 grid(gs_cdiv(H * W, kTcPix), N, num_levels);
    altcorr_tc_kernel<3><<<grid, kTcWarps * 32, 0, (cudaStream_t)stream>>>(a);
  } else {
    dim3 grid(gs_cdiv(H * W, kPixPerBlock), N, num_levels);
    altcorr_pyramid_kernel<3><<<grid, kWarps * 32, smem, (cudaStream_t)stream>>>(a);
  }
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_altcorr_backward(void) { return GOSLAM_EUNSUPPORTED; }

}  // extern "C"
