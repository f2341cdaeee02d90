// conv_tc.cu — the update operator's ConvGRU (SURVEY §8f-4) on tcgen05: 3x3 / 1x1 convolutions as an
// implicit GEMM with the GRU gates fused into the epilogues.
//
// Replaces ConvGRU.forward (src/modules/gru.py:21-39) as called by UpdateModule.forward
// (src/droid_net.py:125, `self.gru(net, inp, corr, flow)`):
//     glo = mean_hw(sigmoid(w(net)) * net)                                   1x1 conv + pooling
//     z = sigmoid(convz([net|inp|corr|flow]) + convz_glo(glo))               3x3, 448 -> 128
//     r = sigmoid(convr([net|inp|corr|flow]) + convr_glo(glo))               3x3, 448 -> 128
//     q = tanh(convq([r*net|inp|corr|flow]) + convq_glo(glo))                3x3, 448 -> 128
//     net' = (1 - z) * net + z * q
// The reference runs 7 cuDNN convolutions, 2 torch.cat of the 448-channel input and ~12 elementwise kernels.
// Here: three launches of ONE kernel (conv_tc_kernel) with different epilogues, plus two tiny ones:
//   pass G  1x1 conv of net, epilogue: sigmoid(.)*net, per-image channel sums       -> glo_sum [B,128]
//   (gru_glo_fc_kernel: the three 128x128 matvecs on the pooled vector              -> glo     [B,384])
//   pass ZR 3x3 conv with z and r stacked to N = 256 (the activation tile is loaded once for both
//           gates), epilogue: bias + glo, sigmoid, z and r*net written                -> z, rnet
//   pass Q  3x3 conv over [rnet|inp|corr|flow], epilogue: tanh, (1-z)*net + z*q       -> net'
//
// Implicit GEMM: M = 128 output pixels (an 8x16 image patch), N = output channels (128 or 256),
// K = taps x input channels in chunks of 64.  Activations are NHWC fp16, so the patch shifted by a tap is ONE
// TMA box (64 ch, 16, 8, 1) of a 4-D tensor map (ch, x, y, image) — image borders are the TMA's zero fill, the
// concatenated input never exists (one tensor map per source tensor) — and lands K-major / SWIZZLE_128B, exactly
// the A operand.  Weights are [tap][cout][cin] fp16: box (64, N, 1) = the B operand.  tcgen05.mma M128 N{128,256}
// K16 accumulates in TMEM (two accumulator stages, so the epilogue of a tile overlaps the MMAs of the next);
// warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..5 = epilogue (one per TMEM lane quadrant).
// fp16 operands, fp32 accumulation, fp32 gate arithmetic, fp16 state — what the reference's autocast region
// computes (src/factor_graph.py:198, torch.cuda.amp.autocast) with one rounding less per gate.
#include "common.cuh"
#include "launch.cuh"
#include "tc_ptx.cuh"

using namespace gs_tc;

namespace {

constexpr int kPY = 8, kPX = 16, kBM = kPY * kPX;   // output patch = MMA M
constexpr int kKC = 64;                             // channels per K chunk (128-byte rows)
constexpr int kABytes = kBM * kKC * 2;              // 16 KB
constexpr int kMaxN = 256;
constexpr int kBBytes = kMaxN * kKC * 2;            // 32 KB (a 128-channel pass uses half)
constexpr int kStages = 4;
constexpr int kThreadsC = 6 * 32;
constexpr int kVecMax = 1024;                       // per-channel epilogue vector (bias, or bias + glo of the tile's image)
constexpr int kSmemC = 1024 + kStages * (kABytes + kBBytes) + 256 + kVecMax * 4;
constexpr int kMaxIn = 4;

enum { EPI_ACT = 0, EPI_GLO = 1, EPI_ZR = 2, EPI_Q = 3 };
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_SIGMOID = 2, ACT_SOFTPLUS = 3 };

struct ConvMaps {
  CUtensorMap in[kMaxIn];
  CUtensorMap w;
};

struct ConvParams {
  int B, h, w, n_yb, n_xb, n_tiles;
  int taps;                 // 1 or 9
  int n_in;
  int chunks[kMaxIn];       // K chunks (64 channels) of each input tensor
  int coff[kMaxIn];         // first channel of each input inside its tensor (a channel slice of a wider NHWC tensor)
  int N;                    // output channels per tile (16..256, multiple of 16)
  int n_nt;                 // output-channel tiles (cout_pad / N)
  // EPI_ACT: out = act(conv + bias) * out_scale, NHWC [.., out_stride] at channel out_offset, first `cout` channels
  int act, cout, out_stride, out_offset, out_f32;
  float out_scale;
  void* out;
  // f32 outputs only: channels >= split go to out2 (same stride) and get act2 instead of act (fused 2-channel heads)
  int split, act2;
  void* out2;
  int epi;
  const float* bias;        // [N]
  const float* glo;         // [B, 384] (z | r | q) or nullptr
  const __half* net;        // [B, h, w, 128] NHWC
  const __half* z_in;       // EPI_Q
  __half* z_out;            // EPI_ZR
  __half* rnet_out;         // EPI_ZR
  __half* net_out;          // EPI_Q
  float* glo_sum;           // EPI_GLO: [B * patches * 4, 128] partial sums over 32 pixels of sigmoid(.) * net
};

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + __expf(-x)); }

// 16 halves = one whole 32-byte sector per store (16-byte pieces are partial-sector writes: read-modify-write in L2)
__device__ __forceinline__ void st_sector(void* dst, const uint32_t (&o)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]),
               "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
}
// 32 values per lane -> lane L returns the sum over lanes of v[L]   (31 shuffles)
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool up = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float send = up ? v[i] : v[i + half];
      const float keep = up ? v[i + half] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  return v[0];
}

__global__ void __launch_bounds__(kThreadsC, 1)
conv_tc_kernel(const __grid_constant__ ConvMaps maps, const ConvParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base =
      reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smA = base;
  unsigned char* smB = base + kStages * kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + kStages * (kABytes + kBBytes));
  uint64_t* full = bars;                    // [kStages]
  uint64_t* empty = full + kStages;         // [kStages]
  uint64_t* tm_full = empty + kStages;      // [2]
  uint64_t* tm_empty = tm_full + 2;         // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tm_empty + 2);
  float* svec = reinterpret_cast<float*>(base + kStages * (kABytes + kBBytes) + 256);   // [kVecMax]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // EPI_ACT / EPI_GLO: the bias vector is the same for every tile: stage it once (per-element global loads inside the
  // epilogue's branches serialised into ~150-cycle waits: ncu long_scoreboard, profiles/r02_conv_notes.md)
  if (p.epi == EPI_ACT || p.epi == EPI_GLO)
    for (int i = threadIdx.x; i < p.n_nt * p.N && i < kVecMax; i += kThreadsC) svec[i] = p.bias[i];
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tm_full[i], 1); mbar_init(&tm_empty[i], 4); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 2 * kMaxN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  int kiters = 0;
  for (int i = 0; i < p.n_in; ++i) kiters += p.chunks[i];
  kiters *= p.taps;
  const uint32_t stage_tx = kABytes + (uint32_t)p.N * kKC * 2;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0, ph = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_nt, pt = tile / p.n_nt;
        const int xb = pt % p.n_xb, yb = (pt / p.n_xb) % p.n_yb, b = pt / (p.n_xb * p.n_yb);
        for (int tap = 0; tap < p.taps; ++tap) {
          const int dy = p.taps == 9 ? tap / 3 - 1 : 0, dx = p.taps == 9 ? tap % 3 - 1 : 0;
          int gchunk = 0;
          for (int ci = 0; ci < p.n_in; ++ci)
            for (int kc = 0; kc < p.chunks[ci]; ++kc, ++gchunk) {
              mbar_wait(&empty[s], ph ^ 1);
              mbar_expect_tx(&full[s], stage_tx);
              tma_load_4d(&maps.in[ci], &full[s], smA + s * kABytes, p.coff[ci] + kc * kKC, xb * kPX + dx, yb * kPY + dy, b);
              tma_load_3d(&maps.w, &full[s], smB + s * kBBytes, gchunk * kKC, nt * p.N, tap);
              if (++s == kStages) { s = 0; ph ^= 1; }
            }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(kBM, p.N);
      int s = 0, ph = 0, ts = 0, tph = 0;
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        mbar_wait(&tm_empty[ts], tph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + ts * kMaxN;
        for (int it = 0; it < kiters; ++it) {
          mbar_wait(&full[s], ph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smA + s * kABytes), b_addr = smem_u32(smB + s * kBBytes);
#pragma unroll
          for (int k = 0; k < kKC / 16; ++k)
            umma_f16(d_tmem, make_desc_sw128(a_addr + k * 32), make_desc_sw128(b_addr + k * 32), idesc,
                     (it | k) != 0 ? 1u : 0u);
          umma_commit(&empty[s]);
          if (++s == kStages) { s = 0; ph ^= 1; }
        }
        umma_commit(&tm_full[ts]);
        if (++ts == 2) { ts = 0; tph ^= 1; }
      }
    }
  } else {
    // ===================== epilogue: warps 2..5, TMEM lane quadrant = warp % 4 =====================
    const int quad = warp & 3;
    const int row = quad * 32 + lane;                // pixel of the patch
    const int py = row / kPX, px = row % kPX;
    int ts = 0, tph = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
      const int nt = tile % p.n_nt, pt = tile / p.n_nt;
      const int xb = pt % p.n_xb, yb = (pt / p.n_xb) % p.n_yb, b = pt / (p.n_xb * p.n_yb);
      const int y = yb * kPY + py, x = xb * kPX + px;
      const bool ok = y < p.h && x < p.w;
      const size_t pix = ((size_t)b * p.h + (ok ? y : 0)) * p.w + (ok ? x : 0);
      if (p.epi == EPI_ZR || p.epi == EPI_Q) {
        // per-tile channel vector = bias + the image's global term, staged by the 128 epilogue threads
        asm volatile("bar.sync 2, 128;" ::: "memory");          // previous tile's vector no longer in use
        const float* glo = p.glo + (size_t)b * 384 + (p.epi == EPI_Q ? 256 : 0);
        for (int i = threadIdx.x - 64; i < p.N; i += 128) svec[i] = p.bias[i] + glo[i];
        asm volatile("bar.sync 2, 128;" ::: "memory");
      }
      mbar_wait(&tm_full[ts], tph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ts * kMaxN + ((uint32_t)(quad * 32) << 16);
      if (p.epi == EPI_ACT) {
        const int act = p.act;
        for (int c0 = 0; c0 < p.N; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(taddr + c0, v);
          const int chb = nt * p.N + c0;             // first output channel of this chunk
          const float* bv = svec + chb;
          float r[32];
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bv + i);
            r[i] = __uint_as_float(v[i]) + b4.x; r[i + 1] = __uint_as_float(v[i + 1]) + b4.y;
            r[i + 2] = __uint_as_float(v[i + 2]) + b4.z; r[i + 3] = __uint_as_float(v[i + 3]) + b4.w;
          }
          if (p.split > 0) {                          // small fused heads (first chunk only holds valid channels)
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (chb + i >= p.split && p.act2 == ACT_SIGMOID) r[i] = sigmoidf_(r[i]);
          }
          if (act == ACT_RELU) {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = fmaxf(r[i], 0.f);
          } else if (act == ACT_SIGMOID) {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = sigmoidf_(r[i]);
          } else if (act == ACT_SOFTPLUS) {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = (r[i] > 20.f) ? r[i] : log1pf(__expf(r[i]));
          }
          if (p.out_scale != 1.0f) {
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] *= p.out_scale;
          }
          if (ok) {
            if (p.out_f32) {
              float* dst = reinterpret_cast<float*>(p.out) + pix * p.out_stride + p.out_offset + chb;
              float* dst2 = reinterpret_cast<float*>(p.out2) + pix * p.out_stride - p.split + chb;
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c0 + i < p.N && chb + i < p.cout) {
                  if (p.split > 0 && chb + i >= p.split) dst2[i] = r[i];
                  else dst[i] = r[i];
                }
            } else {
              __half* dst = reinterpret_cast<__half*>(p.out) + pix * p.out_stride + p.out_offset + chb;
#pragma unroll
              for (int i = 0; i < 32; i += 16) {
                if (c0 + i + 16 <= p.N && chb + i + 16 <= p.cout && ((p.out_stride | (p.out_offset + chb + i)) & 15) == 0) {
                  uint32_t o[8];
#pragma unroll
                  for (int k = 0; k < 8; ++k) {
                    const __half2 hv = __floats2half2_rn(r[i + 2 * k], r[i + 2 * k + 1]);
                    o[k] = *reinterpret_cast<const uint32_t*>(&hv);
                  }
                  st_sector(dst + i, o);
                } else {
#pragma unroll
                  for (int k = 0; k < 16; ++k)
                    if (c0 + i + k < p.N && chb + i + k < p.cout) dst[i + k] = __float2half_rn(r[i + k]);
                }
              }
            }
          }
        }
      } else
      for (int c0 = 0; c0 < p.N; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + c0, v);
        const int ch = c0 & 127;                     // channel of the 128-channel state this chunk maps to
        uint4 netv[4];
        if (ok) {
          const uint4* np = reinterpret_cast<const uint4*>(p.net + pix * 128 + ch);
#pragma unroll
          for (int i = 0; i < 4; ++i) netv[i] = __ldg(np + i);
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) netv[i] = make_uint4(0, 0, 0, 0);
        }
        const __half2* nh = reinterpret_cast<const __half2*>(netv);
        float a[32];                                  // accumulator + per-channel vector (bias [+ glo])
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 b4 = *reinterpret_cast<const float4*>(svec + c0 + i);
          a[i] = __uint_as_float(v[i]) + b4.x; a[i + 1] = __uint_as_float(v[i + 1]) + b4.y;
          a[i + 2] = __uint_as_float(v[i + 2]) + b4.z; a[i + 3] = __uint_as_float(v[i + 3]) + b4.w;
        }
        if (p.epi == EPI_GLO) {
          // g = sigmoid(conv + b) * net; per-image channel sums (the mean's divisor is applied by the fc kernel)
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float nv = (i & 1) ? __high2float(nh[i >> 1]) : __low2float(nh[i >> 1]);
            a[i] = ok ? sigmoidf_(a[i]) * nv : 0.f;
          }
          const float tot = warp_transpose_sum32(a, lane);      // lane L: sum over the warp's 32 pixels of channel c0+L
          p.glo_sum[((size_t)pt * 4 + quad) * 128 + c0 + lane] = tot;   // one partial per (patch, warp): deterministic
        } else if (p.epi == EPI_ZR) {
          const bool is_r = c0 >= 128;
          uint32_t o[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float g0 = sigmoidf_(a[i]), g1 = sigmoidf_(a[i + 1]);
            const float2 nv = __half22float2(nh[i >> 1]);
            const __half2 h = is_r ? __floats2half2_rn(g0 * nv.x, g1 * nv.y) : __floats2half2_rn(g0, g1);
            o[i >> 1] = *reinterpret_cast<const uint32_t*>(&h);
          }
          if (ok) {
            __half* dst = (is_r ? p.rnet_out : p.z_out) + pix * 128 + ch;
            const uint32_t (&lo)[8] = *reinterpret_cast<const uint32_t (*)[8]>(&o[0]);
            const uint32_t (&hi)[8] = *reinterpret_cast<const uint32_t (*)[8]>(&o[8]);
            st_sector(dst, lo);
            st_sector(dst + 16, hi);
          }
        } else {   // EPI_Q
          uint4 zv[4];
          if (ok) {
            const uint4* zp = reinterpret_cast<const uint4*>(p.z_in + pix * 128 + ch);
#pragma unroll
            for (int i = 0; i < 4; ++i) zv[i] = __ldg(zp + i);
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) zv[i] = make_uint4(0, 0, 0, 0);
          }
          const __half2* zh = reinterpret_cast<const __half2*>(zv);
          uint32_t o[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            const float q0 = tanhf(a[i]), q1 = tanhf(a[i + 1]);
            const float2 nv = __half22float2(nh[i >> 1]), zz = __half22float2(zh[i >> 1]);
            const __half2 h = __floats2half2_rn((1.0f - zz.x) * nv.x + zz.x * q0, (1.0f - zz.y) * nv.y + zz.y * q1);
            o[i >> 1] = *reinterpret_cast<const uint32_t*>(&h);
          }
          if (ok) {
            __half* dst = p.net_out + pix * 128 + ch;
            const uint32_t (&lo)[8] = *reinterpret_cast<const uint32_t (*)[8]>(&o[0]);
            const uint32_t (&hi)[8] = *reinterpret_cast<const uint32_t (*)[8]>(&o[8]);
            st_sector(dst, lo);
            st_sector(dst + 16, hi);
          }
        }
      }
      // all TMEM reads of this warp for this stage are complete (tmem_ld32 waits): hand the stage back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tm_empty[ts]);
      if (++ts == 2) { ts = 0; tph ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * kMaxN);
}

// glo[b] = W_glo mean_px(sigmoid(w(net)) * net) + b_glo : sums the per-(patch, warp) partials of pass G in a fixed order,
// then the three 1x1 "global" convolutions on the pooled vector, one warp per output (coalesced weight rows)
__global__ void __launch_bounds__(256)
gru_glo_fc_kernel(const float* __restrict__ part, int parts_per_image, const float* __restrict__ w_glo,
                  const float* __restrict__ b_glo, float* __restrict__ glo, float inv_hw) {
  __shared__ float v[128];
  const int b = blockIdx.x;
  if (threadIdx.x < 128) {
    const float* pp = part + (size_t)b * parts_per_image * 128 + threadIdx.x;
    float acc = 0.f;
    for (int i = 0; i < parts_per_image; ++i) acc += pp[(size_t)i * 128];
    v[threadIdx.x] = acc * inv_hw;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int o = warp; o < 384; o += 8) {
    const float4 wv = *reinterpret_cast<const float4*>(w_glo + (size_t)o * 128 + lane * 4);
    float acc = wv.x * v[lane * 4] + wv.y * v[lane * 4 + 1] + wv.z * v[lane * 4 + 2] + wv.w * v[lane * 4 + 3];
    acc = gs_warp_sum(acc);
    if (lane == 0) glo[(size_t)b * 384 + o] = acc + b_glo[o];
  }
}

// [B, rows, cols] -> [B, cols, rows] fp16 through a 32x32 shared-memory tile (generic shapes)
__global__ void transpose_f16_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int rows, int cols) {
  __shared__ __half t[32][34];
  const size_t boff = (size_t)blockIdx.z * rows * cols;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    if (r < rows && c < cols) t[i][threadIdx.x] = src[boff + (size_t)r * cols + c];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < rows && c < cols) dst[boff + (size_t)c * rows + r] = t[threadIdx.x][i];
  }
}

// Fast path of the two layout conversions, 64 x 64 tiles: 16-byte loads along the source's contiguous dimension, whole
// 32-byte sectors (16 halves) on the way out, both shared-memory phases conflict-free (row stride 33 words).
//   NCHW -> NHWC: src [B][C][hw] (rows = channels, zero beyond C), dst [B][hw][Cpad]
__global__ void __launch_bounds__(256)
nchw_to_nhwc64_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int C, int Cpad, int hw) {
  __shared__ uint32_t t[64][33];
  const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 64;          // r: channel, c: pixel
  const __half* s = src + (size_t)blockIdx.z * C * hw;
  __half* d = dst + (size_t)blockIdx.z * hw * Cpad;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int idx = threadIdx.x + 256 * i, r = idx >> 3, c8 = idx & 7;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (r0 + r < C && c0 + c8 * 8 < hw) v = __ldg(reinterpret_cast<const uint4*>(s + (size_t)(r0 + r) * hw + c0 + c8 * 8));
    t[r][c8 * 4 + 0] = v.x; t[r][c8 * 4 + 1] = v.y; t[r][c8 * 4 + 2] = v.z; t[r][c8 * 4 + 3] = v.w;
  }
  __syncthreads();
  const int px = threadIdx.x & 63, r16 = threadIdx.x >> 6;
  if (c0 + px < hw && r0 + r16 * 16 < Cpad) {
    uint32_t o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t a = t[r16 * 16 + 2 * j][px >> 1], b = t[r16 * 16 + 2 * j + 1][px >> 1];
      const uint32_t lo = (px & 1) ? (a >> 16) : (a & 0xffffu), hi = (px & 1) ? (b >> 16) : (b & 0xffffu);
      o[j] = lo | (hi << 16);
    }
    st_sector(d + (size_t)(c0 + px) * Cpad + r0 + r16 * 16, o);
  }
}
//   NHWC -> NCHW: src [B][hw][C] (C % 64 == 0), dst [B][C][hw]; rows = pixels here
__global__ void __launch_bounds__(256)
nhwc_to_nchw64_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int C, int hw) {
  __shared__ uint32_t t[64][33];
  const int p0 = blockIdx.y * 64, c0 = blockIdx.x * 64;          // rows: pixel, cols: channel
  const __half* s = src + (size_t)blockIdx.z * hw * C;
  __half* d = dst + (size_t)blockIdx.z * C * hw;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int idx = threadIdx.x + 256 * i, r = idx >> 3, c8 = idx & 7;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (p0 + r < hw) v = __ldg(reinterpret_cast<const uint4*>(s + (size_t)(p0 + r) * C + c0 + c8 * 8));
    t[r][c8 * 4 + 0] = v.x; t[r][c8 * 4 + 1] = v.y; t[r][c8 * 4 + 2] = v.z; t[r][c8 * 4 + 3] = v.w;
  }
  __syncthreads();
  const int ch = threadIdx.x & 63, q16 = threadIdx.x >> 6;        // 16 consecutive pixels of one channel
  if (p0 + q16 * 16 < hw) {
    uint32_t o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t a = t[q16 * 16 + 2 * j][ch >> 1], b = t[q16 * 16 + 2 * j + 1][ch >> 1];
      const uint32_t lo = (ch & 1) ? (a >> 16) : (a & 0xffffu), hi = (ch & 1) ? (b >> 16) : (b & 0xffffu);
      o[j] = lo | (hi << 16);
    }
    __half* dp = d + (size_t)(c0 + ch) * hw + p0 + q16 * 16;
    if (p0 + q16 * 16 + 16 <= hw) st_sector(dp, o);
    else
      for (int j = 0; j < 16 && p0 + q16 * 16 + j < hw; ++j)
        dp[j] = __ushort_as_half((unsigned short)((o[j >> 1] >> ((j & 1) * 16)) & 0xffffu));
  }
}

// [B, C, hw] -> [B, hw, Cpad] with zero channels C..Cpad-1
__global__ void transpose_pad_f16_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int C, int Cpad, int hw) {
  __shared__ __half t[32][34];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;          // r: channel, c: pixel
  const __half* s = src + (size_t)blockIdx.z * C * hw;
  __half* d = dst + (size_t)blockIdx.z * hw * Cpad;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    t[i][threadIdx.x] = (r < C && c < hw) ? s[(size_t)r * hw + c] : __half(0.f);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < Cpad && c < hw) d[(size_t)c * Cpad + r] = t[threadIdx.x][i];
  }
}

// flow_encoder.0 (src/droid_net.py:84): 7x7 convolution of the 4 motion channels to 128 + ReLU.  K = 196 is too thin for
// the tensor-core path's 64-channel chunks; CUDA cores: block = 8x16 output patch, thread = (pixel, half of the output
// channels), the 14x22x4 input halo and the [196][128] weights (fp32) in shared memory, 64 accumulators per thread.
//   in  [B,4,h,w] f32 (the motion features as FactorGraph hands them over), out [B,h,w,128] f16 NHWC
constexpr int kF7Halo = (kPY + 6) * (kPX + 6) * 4;
__global__ void __launch_bounds__(256)
flow7x7_kernel(const float* __restrict__ in, const float* __restrict__ wgt /*[196][128]: k = (ky*7+kx)*4+ci*/,
               const float* __restrict__ bias, __half* __restrict__ out, int h, int w) {
  extern __shared__ float sm7[];
  float* sw = sm7;                       // [196][128]
  float* si = sm7 + 196 * 128;           // [14][22][4]
  const int n_xb = gs_cdiv_dev(w, kPX), n_yb = gs_cdiv_dev(h, kPY);
  const int xb = blockIdx.x % n_xb, yb = (blockIdx.x / n_xb) % n_yb, b = blockIdx.x / (n_xb * n_yb);
  for (int i = threadIdx.x; i < 196 * 128; i += 256) sw[i] = wgt[i];
  for (int i = threadIdx.x; i < kF7Halo; i += 256) {
    const int ci = i & 3, xx = (i >> 2) % (kPX + 6), yy = (i >> 2) / (kPX + 6);
    const int gx = xb * kPX + xx - 3, gy = yb * kPY + yy - 3;
    si[i] = (gx >= 0 && gx < w && gy >= 0 && gy < h) ? in[(((size_t)b * 4 + ci) * h + gy) * w + gx] : 0.f;
  }
  __syncthreads();
  const int pix = threadIdx.x & 127, chh = threadIdx.x >> 7;      // 64 output channels each
  const int py = pix / kPX, px = pix % kPX;
  float acc[64];
#pragma unroll
  for (int c = 0; c < 64; ++c) acc[c] = bias[chh * 64 + c];
  for (int ky = 0; ky < 7; ++ky)
    for (int kx = 0; kx < 7; ++kx) {
      const float4 v = *reinterpret_cast<const float4*>(si + ((py + ky) * (kPX + 6) + px + kx) * 4);
      const float* wr = sw + ((ky * 7 + kx) * 4) * 128 + chh * 64;
#pragma unroll
      for (int c = 0; c < 64; c += 4) {
        const float4 w0 = *reinterpret_cast<const float4*>(wr + c);
        const float4 w1 = *reinterpret_cast<const float4*>(wr + 128 + c);
        const float4 w2 = *reinterpret_cast<const float4*>(wr + 256 + c);
        const float4 w3 = *reinterpret_cast<const float4*>(wr + 384 + c);
        acc[c] += v.x * w0.x + v.y * w1.x + v.z * w2.x + v.w * w3.x;
        acc[c + 1] += v.x * w0.y + v.y * w1.y + v.z * w2.y + v.w * w3.y;
        acc[c + 2] += v.x * w0.z + v.y * w1.z + v.z * w2.z + v.w * w3.z;
        acc[c + 3] += v.x * w0.w + v.y * w1.w + v.z * w2.w + v.w * w3.w;
      }
    }
  const int y = yb * kPY + py, x = xb * kPX + px;
  if (y < h && x < w) {
    __half* dst = out + (((size_t)b * h + y) * w + x) * 128 + chh * 64;
#pragma unroll
    for (int c = 0; c < 64; c += 8) {
      __half2 hv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) hv[j] = __floats2half2_rn(fmaxf(acc[c + 2 * j], 0.f), fmaxf(acc[c + 2 * j + 1], 0.f));
      *reinterpret_cast<uint4*>(dst + c) = *reinterpret_cast<const uint4*>(hv);
    }
  }
}

// Tensor-core version: im2col in shared memory.  K = 49 taps x 4 channels = 196, zero-padded to 256 = four 64-wide
// chunks.  The 128 builder threads (one per output pixel of the 8x16 patch) write their im2col row straight into the
// K-major SWIZZLE_128B operand layout the TMA would have produced (row r of a chunk at r*128 B inside 8-row / 1024-byte
// atoms, its 16-byte pieces XOR-ed with r % 8); the weights [128][256] come in once per CTA by TMA; 16 tcgen05.mma
// (M128 N128 K16) per tile; bias + ReLU epilogue to NHWC f16.
constexpr int kF7K = 256, kF7ABytes = kBM * kF7K * 2, kF7BBytes = 128 * kF7K * 2;
constexpr int kF7Smem = 1024 + kF7ABytes + kF7BBytes + kF7Halo * 4 + 128 * 4 + 256;
__global__ void __launch_bounds__(160, 1)
flow7x7_tc_kernel(const __grid_constant__ CUtensorMap wmap, const float* __restrict__ in, const float* __restrict__ bias,
                  __half* __restrict__ out, int B, int h, int w) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base =
      reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smA = base;
  unsigned char* smB = base + kF7ABytes;
  float* si = reinterpret_cast<float*>(smB + kF7BBytes);          // [14][22][4]
  float* sb = si + kF7Halo;                                       // [128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sb + 128);
  uint64_t* w_full = bars;
  uint64_t* mma_done = bars + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { mbar_init(w_full, 1); mbar_init(mma_done, 1); fence_barrier_init(); }
  if (warp == 4) tmem_alloc(tmem_ptr, 128);
  for (int i = threadIdx.x; i < 128; i += 160) sb[i] = bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  if (threadIdx.x == 128) {                          // weights: four (64 K, 128 cout) boxes, once
    mbar_expect_tx(w_full, kF7BBytes);
    for (int kc = 0; kc < 4; ++kc) tma_load_3d(&wmap, w_full, smB + kc * (128 * 128), kc * 64, 0, 0);
  }
  const int n_xb = gs_cdiv_dev(w, kPX), n_yb = gs_cdiv_dev(h, kPY), n_tiles = B * n_xb * n_yb;
  uint32_t ph = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int xb = tile % n_xb, yb = (tile / n_xb) % n_yb, b = tile / (n_xb * n_yb);
    // ---- input halo (fp32), all threads
    for (int i = threadIdx.x; i < kF7Halo; i += 160) {
      const int ci = i & 3, xx = (i >> 2) % (kPX + 6), yy = (i >> 2) / (kPX + 6);
      const int gx = xb * kPX + xx - 3, gy = yb * kPY + yy - 3;
      si[i] = (gx >= 0 && gx < w && gy >= 0 && gy < h) ? in[(((size_t)b * 4 + ci) * h + gy) * w + gx] : 0.f;
    }
    __syncthreads();
    // ---- im2col rows into the swizzled A tile
    if (threadIdx.x < 128) {
      const int r = threadIdx.x, py = r / kPX, px = r % kPX;
      unsigned char* rowp = smA + (r >> 3) * 1024 + (r & 7) * 128;
      for (int t2 = 0; t2 < 32; ++t2) {              // pairs of taps = one 16-byte piece (8 halves)
        uint32_t o[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int t = 2 * t2 + u;
          if (t < 49) {
            const float4 v = *reinterpret_cast<const float4*>(si + ((py + t / 7) * (kPX + 6) + px + t % 7) * 4);
            const __half2 a = __floats2half2_rn(v.x, v.y), c = __floats2half2_rn(v.z, v.w);
            o[2 * u] = *reinterpret_cast<const uint32_t*>(&a);
            o[2 * u + 1] = *reinterpret_cast<const uint32_t*>(&c);
          }
        }
        const int kc = t2 >> 3, c16 = t2 & 7;
        *reinterpret_cast<uint4*>(rowp + kc * (kBM * 128) + ((c16 ^ (r & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
    fence_async_smem();                              // generic-proxy writes -> visible to the tensor core (async proxy)
    __syncthreads();
    if (threadIdx.x == 128) {
      if (tile == (int)blockIdx.x) mbar_wait(w_full, 0);
      tc_fence_after();
      const uint32_t idesc = make_idesc_f16(kBM, 128);
      const uint32_t a_addr = smem_u32(smA), b_addr = smem_u32(smB);
#pragma unroll
      for (int kc = 0; kc < 4; ++kc)
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_f16(tmem_base, make_desc_sw128(a_addr + kc * (kBM * 128) + k * 32), make_desc_sw128(b_addr + kc * (128 * 128) + k * 32),
                   idesc, (kc | k) != 0 ? 1u : 0u);
      umma_commit(mma_done);
    }
    // ---- epilogue: warps 0..3 = TMEM lane quadrants
    if (threadIdx.x < 128) {
      mbar_wait(mma_done, ph);
      tc_fence_after();
      const int r = threadIdx.x, py = r / kPX, px = r % kPX;
      const int y = yb * kPY + py, x = xb * kPX + px;
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + c0, v);
        if (y < h && x < w) {
          __half* dst = out + (((size_t)b * h + y) * w + x) * 128 + c0;
#pragma unroll
          for (int i = 0; i < 32; i += 16) {
            uint32_t o[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const __half2 hv = __floats2half2_rn(fmaxf(__uint_as_float(v[i + 2 * k]) + sb[c0 + i + 2 * k], 0.f),
                                                   fmaxf(__uint_as_float(v[i + 2 * k + 1]) + sb[c0 + i + 2 * k + 1], 0.f));
              o[k] = *reinterpret_cast<const uint32_t*>(&hv);
            }
            st_sector(dst + i, o);
          }
        }
      }
      tc_fence_before();
    }
    ph ^= 1;
    __syncthreads();                                 // A tile, halo and TMEM free for the next tile
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 128);
}

// GraphAgg's scatter_mean (src/droid_net.py:59): mean over the edges of each source frame, NHWC f16, fp32 sums in edge
// order (deterministic).  thread = (frame slot m, pixel, 8-channel chunk)
__global__ void __launch_bounds__(256)
scatter_mean_kernel(const __half* __restrict__ a1, const int* __restrict__ slot, __half* __restrict__ mean, int N, int M,
                    int hw) {
  const size_t t = (size_t)blockIdx.x * 256 + threadIdx.x;
  const size_t total = (size_t)M * hw * 16;
  if (t >= total) return;
  const int c8 = (int)(t & 15);
  const size_t px = (t >> 4) % hw;
  const int m = (int)((t >> 4) / hw);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  int cnt = 0;
  for (int e = 0; e < N; ++e) {
    if (__ldg(slot + e) != m) continue;
    ++cnt;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(a1 + ((size_t)e * hw + px) * 128 + c8 * 8));
    const __half2* hv = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(hv[j]); acc[2 * j] += f.x; acc[2 * j + 1] += f.y; }
  }
  const float inv = cnt > 0 ? 1.0f / (float)cnt : 0.f;
  __half2 o[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) o[j] = __floats2half2_rn(acc[2 * j] * inv, acc[2 * j + 1] * inv);
  *reinterpret_cast<uint4*>(mean + ((size_t)m * hw + px) * 128 + c8 * 8) = *reinterpret_cast<const uint4*>(o);
}

// Tensor maps depend only on (base pointer, shape): the update operator runs the same layers on the same workspace
// buffers call after call, so the encodes (~50 per operator call) are paid once.
enum { kActMap = 0, kWeightMap = 1 };

bool encode_cmap(GsEncodeTiledFn enc, const GsMapKey& k, CUtensorMap* out) {
  if (k.kind == kActMap) {
    // activation map: NHWC [B, h, w, C] as (ch, x, y, image), box 64 ch x 16 x 8
    const int B = k.dims[0], h = k.dims[1], w = k.dims[2], C = k.dims[3];
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)w * C * 2, (cuuint64_t)h * w * C * 2};
    cuuint32_t box[4] = {(cuuint32_t)kKC, (cuuint32_t)kPX, (cuuint32_t)kPY, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(k.base), dims, strides, box, es,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  // weight map: [taps, N, Cin] as (cin, cout, tap), box 64 x n_tile (0: N)
  const int taps = k.dims[0], N = k.dims[1], Cin = k.dims[2], n_tile = k.dims[3];
  cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)N, (cuuint64_t)taps};
  cuuint64_t strides[2] = {(cuuint64_t)Cin * 2, (cuuint64_t)N * Cin * 2};
  cuuint32_t box[3] = {(cuuint32_t)kKC, (cuuint32_t)(n_tile > 0 ? n_tile : N), 1};
  cuuint32_t es[3] = {1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(k.base), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

GsMapCache g_cmaps(128, encode_cmap);

bool act_map(const void* base, int B, int h, int w, int C, CUtensorMap* out) {
  return g_cmaps.get(GsMapKey{base, kActMap, {B, h, w, C}}, out);
}
bool weight_map(const void* base, int taps, int N, int Cin, CUtensorMap* out, int n_tile = 0) {
  return g_cmaps.get(GsMapKey{base, kWeightMap, {taps, N, Cin, n_tile}}, out);
}

GsDeviceOnce g_conv_once;
cudaError_t conv_device_init(int) {
  cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemC);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(flow7x7_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kF7Smem);
  return e;
}

int conv_launch(const ConvMaps& maps, ConvParams p, cudaStream_t st) {
  const int rc = gs_device_once(g_conv_once, conv_device_init);
  if (rc != GOSLAM_OK) return rc;
  const int sms = gs_sm_count();
  p.n_yb = gs_cdiv(p.h, kPY); p.n_xb = gs_cdiv(p.w, kPX);
  if (p.n_nt < 1) p.n_nt = 1;
  p.n_tiles = p.B * p.n_yb * p.n_xb * p.n_nt;
  const int grid = p.n_tiles < sms ? p.n_tiles : sms;
  conv_tc_kernel<<<grid, kThreadsC, kSmemC, st>>>(maps, p);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

struct GruWs {
  float* glo_sum;   // [B,128]
  float* glo;       // [B,384]
  __half* z;        // [B,h,w,128]
  __half* rnet;     // [B,h,w,128]
};
size_t gru_layout(int B, int h, int w, void* base, size_t cap, GruWs* ws) {
  GsArena a(base, cap);
  GruWs g{};
  g.glo_sum = a.take<float>((size_t)B * gs_cdiv(h, kPY) * gs_cdiv(w, kPX) * 4 * 128);
  g.glo = a.take<float>((size_t)B * 384);
  g.z = a.take<__half>((size_t)B * h * w * 128);
  g.rnet = a.take<__half>((size_t)B * h * w * 128);
  if (ws) *ws = g;
  return a.off;
}

}  // namespace

extern "C" {

int goslam_nchw_to_nhwc_f16(const void* src, void* dst, int B, int C, int hw, void* stream) {
  if (B < 0 || C <= 0 || hw <= 0) return GOSLAM_EINVAL;
  if (B == 0) return GOSLAM_OK;
  if (hw % 16 == 0 && C % 16 == 0) {
    nchw_to_nhwc64_kernel<<<dim3(gs_cdiv(hw, 64), gs_cdiv(C, 64), B), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __half*>(src), reinterpret_cast<__half*>(dst), C, C, hw);
    GS_CHECK_LAUNCH();
    return GOSLAM_OK;
  }
  dim3 grid(gs_cdiv(hw, 32), gs_cdiv(C, 32), B), block(32, 8);
  transpose_f16_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __half*>(src),
                                                                  reinterpret_cast<__half*>(dst), C, hw);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_nhwc_to_nchw_f16(const void* src, void* dst, int B, int C, int hw, void* stream) {
  if (B < 0 || C <= 0 || hw <= 0) return GOSLAM_EINVAL;
  if (B == 0) return GOSLAM_OK;
  if (hw % 16 == 0 && C % 64 == 0) {
    nhwc_to_nchw64_kernel<<<dim3(C / 64, gs_cdiv(hw, 64), B), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __half*>(src), reinterpret_cast<__half*>(dst), C, hw);
    GS_CHECK_LAUNCH();
    return GOSLAM_OK;
  }
  dim3 grid(gs_cdiv(C, 32), gs_cdiv(hw, 32), B), block(32, 8);
  transpose_f16_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __half*>(src),
                                                                  reinterpret_cast<__half*>(dst), hw, C);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_conv2d_nhwc(const goslam_conv_desc* d, int B, int h, int w, void* stream) {
  if (!d || B < 0 || h <= 0 || w <= 0 || d->n_in < 1 || d->n_in > kMaxIn) return GOSLAM_EINVAL;
  if ((d->taps != 1 && d->taps != 9) || d->cout < 1 || d->cout_pad < d->cout || d->cout_pad % 16) return GOSLAM_EINVAL;
  const int N = d->cout_pad <= kMaxN ? d->cout_pad : (d->cout_pad % 192 == 0 ? 192 : (d->cout_pad % 256 == 0 ? 256 : 128));
  if (d->cout_pad % N) return GOSLAM_EINVAL;
  if (B == 0) return GOSLAM_OK;
  ConvMaps m{};
  ConvParams p{};
  p.B = B; p.h = h; p.w = w; p.taps = d->taps; p.n_in = d->n_in; p.N = N; p.n_nt = d->cout_pad / N;
  int cin_total = 0;
  for (int i = 0; i < d->n_in; ++i) {
    if (d->cin[i] <= 0 || d->cin[i] % kKC || d->cin_off[i] % kKC || d->cin_stride[i] < d->cin_off[i] + d->cin[i]) return GOSLAM_EINVAL;
    p.chunks[i] = d->cin[i] / kKC; p.coff[i] = d->cin_off[i];
    cin_total += d->cin[i];
    if (!act_map(d->in[i], B, h, w, d->cin_stride[i], &m.in[i])) return GOSLAM_ELAUNCH;
  }
  if (!weight_map(d->weight, d->taps, d->cout_pad, cin_total, &m.w, N)) return GOSLAM_ELAUNCH;
  p.epi = EPI_ACT; p.bias = d->bias; p.act = d->act; p.cout = d->cout; p.out = d->out; p.out_f32 = d->out_f32;
  p.out_stride = d->out_stride; p.out_offset = d->out_offset; p.out_scale = d->out_scale;
  p.split = d->split; p.act2 = d->act2; p.out2 = d->out2;
  if (d->split > 0 && (!d->out_f32 || !d->out2 || d->cout > 8)) return GOSLAM_EINVAL;
  if (!d->out_f32 && ((d->out_stride % 8) || (d->out_offset % 8))) return GOSLAM_EINVAL;
  return conv_launch(m, p, (cudaStream_t)stream);
}

int goslam_nchw_to_nhwc_f16_pad(const void* src, void* dst, int B, int C, int Cpad, int hw, void* stream) {
  if (B < 0 || C <= 0 || Cpad < C || hw <= 0) return GOSLAM_EINVAL;
  if (B == 0) return GOSLAM_OK;
  if (hw % 16 == 0 && Cpad % 16 == 0 && hw % 8 == 0) {
    nchw_to_nhwc64_kernel<<<dim3(gs_cdiv(hw, 64), gs_cdiv(Cpad, 64), B), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const __half*>(src), reinterpret_cast<__half*>(dst), C, Cpad, hw);
    GS_CHECK_LAUNCH();
    return GOSLAM_OK;
  }
  dim3 grid(gs_cdiv(hw, 32), gs_cdiv(Cpad, 32), B), block(32, 8);
  transpose_pad_f16_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __half*>(src),
                                                                      reinterpret_cast<__half*>(dst), C, Cpad, hw);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

size_t goslam_conv_gru_workspace_bytes(int B, int h, int w) {
  if (B <= 0 || h <= 0 || w <= 0) return 256;
  return gru_layout(B, h, w, nullptr, 0, nullptr) + 256;
}

// ------------------------------------------------------------------------------------------------------
// The whole update operator in one call (UpdateModule.forward, src/droid_net.py:107-140): layout conversion of the
// reference-shaped inputs, encoders, ConvGRU, heads, GraphAgg — ~20 launches issued from here, tensor maps cached.
// ------------------------------------------------------------------------------------------------------
struct OpWs {
  __half *corr256, *c1, *c2, *f1, *f2, *net, *inp, *state, *hid, *a1, *mean, *a2, *up;
  void* gru;
  size_t gru_bytes;
};
static size_t op_layout(int N, int M, int h, int w, void* base, size_t cap, OpWs* out) {
  GsArena a(base, cap);
  OpWs o{};
  const size_t px = (size_t)N * h * w, pm = (size_t)(M > 0 ? M : 1) * h * w;
  o.corr256 = a.take<__half>(px * 256); o.c1 = a.take<__half>(px * 128); o.c2 = a.take<__half>(px * 128);
  o.f1 = a.take<__half>(px * 128); o.f2 = a.take<__half>(px * 64);
  o.net = a.take<__half>(px * 128); o.inp = a.take<__half>(px * 128); o.state = a.take<__half>(px * 128);
  o.hid = a.take<__half>(px * 256); o.a1 = a.take<__half>(px * 128);
  o.mean = a.take<__half>(pm * 128); o.a2 = a.take<__half>(pm * 128); o.up = a.take<__half>(pm * 576);
  o.gru_bytes = goslam_conv_gru_workspace_bytes(N, h, w);
  o.gru = a.take<char>(o.gru_bytes);
  if (out) *out = o;
  return a.off;
}

static int layer(const void* in, int cin, int cin_off, int cin_stride, const void* wgt, const float* bias, int taps, int cout,
          int cout_pad, int act, float scale, void* out, int out_f32, int out_stride, int B, int h, int w, void* stream) {
  goslam_conv_desc d{};
  d.in[0] = in; d.cin[0] = cin; d.cin_off[0] = cin_off; d.cin_stride[0] = cin_stride; d.n_in = 1;
  d.weight = wgt; d.bias = bias; d.taps = taps; d.cout = cout; d.cout_pad = cout_pad; d.act = act; d.out_scale = scale;
  d.out = out; d.out_f32 = out_f32; d.out_stride = out_stride; d.out_offset = 0;
  return goslam_conv2d_nhwc(&d, B, h, w, stream);
}

size_t goslam_update_op_workspace_bytes(int N, int M, int h, int w) {
  if (N <= 0 || h <= 0 || w <= 0) return 256;
  return op_layout(N, M, h, w, nullptr, 0, nullptr) + 256;
}

int goslam_update_op(const goslam_update_weights* W, const void* net, const void* inp, const void* corr,
                     const float* flow, const int* frame_slot, int N, int M, int h, int w, void* net_out,
                     float* delta, float* weight, float* eta, void* upmask, void* workspace,
                     size_t workspace_bytes, void* stream) {
  if (!W || N < 0 || h <= 0 || w <= 0 || (frame_slot && M <= 0)) return GOSLAM_EINVAL;
  if (N == 0) return GOSLAM_OK;
  OpWs ws;
  const size_t need = op_layout(N, frame_slot ? M : 0, h, w, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int hw = h * w;
  int rc;
#define GS_TRY(x) do { rc = (x); if (rc) return rc; } while (0)
  // ---- reference-shaped inputs ([N,C,h,w]) -> NHWC f16
  GS_TRY(goslam_nchw_to_nhwc_f16_pad(corr, ws.corr256, N, 196, 256, hw, stream));
  GS_TRY(goslam_nchw_to_nhwc_f16(net, ws.net, N, 128, hw, stream));
  GS_TRY(goslam_nchw_to_nhwc_f16(inp, ws.inp, N, 128, hw, stream));
  // ---- encoders (src/droid_net.py:76-88)
  GS_TRY(layer(ws.corr256, 256, 0, 256, W->corr0_w, W->corr0_b, 1, 128, 128, ACT_RELU, 1.f, ws.c1, 0, 128, N, h, w, stream));
  GS_TRY(layer(ws.c1, 128, 0, 128, W->corr2_w, W->corr2_b, 9, 128, 128, ACT_RELU, 1.f, ws.c2, 0, 128, N, h, w, stream));
  {
    // 7x7 motion encoder: im2col + tcgen05 (flow0_w f16 [128][256], K = (ky*7+kx)*4 + ci, zero beyond 196)
    CUtensorMap wm;
    if (!weight_map(W->flow0_w, 1, 128, kF7K, &wm, 128)) return GOSLAM_ELAUNCH;
    GS_TRY(gs_device_once(g_conv_once, conv_device_init));
    const int sms = gs_sm_count();
    const int n_tiles = N * gs_cdiv(h, kPY) * gs_cdiv(w, kPX);
    flow7x7_tc_kernel<<<n_tiles < sms ? n_tiles : sms, 160, kF7Smem, st>>>(wm, flow, W->flow0_b, ws.f1, N, h, w);
    GS_CHECK_LAUNCH();
  }
  GS_TRY(layer(ws.f1, 128, 0, 128, W->flow2_w, W->flow2_b, 9, 64, 64, ACT_RELU, 1.f, ws.f2, 0, 64, N, h, w, stream));
  // ---- ConvGRU
  GS_TRY(goslam_conv_gru(&W->gru, ws.net, ws.inp, ws.c2, ws.f2, ws.state, N, h, w, ws.gru, ws.gru_bytes, stream));
  // ---- heads: delta.0 | weight.0 stacked (shared input), then the two 2-channel heads on their halves, fp32 out
  GS_TRY(layer(ws.state, 128, 0, 128, W->hid_w, W->hid_b, 9, 256, 256, ACT_RELU, 1.f, ws.hid, 0, 256, N, h, w, stream));
  {
    // delta.2 and weight.2 in ONE pass over the 256 hidden channels with block-diagonal weights
    // (heads_w [9][16][256]: row 0-1 = delta.2 on channels 0..127, rows 2-3 = weight.2 on channels 128..255)
    goslam_conv_desc d{};
    d.in[0] = ws.hid; d.cin[0] = 256; d.cin_off[0] = 0; d.cin_stride[0] = 256; d.n_in = 1;
    d.weight = W->delta_w; d.bias = W->delta_b; d.taps = 9; d.cout = 4; d.cout_pad = 16; d.act = ACT_NONE; d.out_scale = 1.f;
    d.out = delta; d.out_f32 = 1; d.out_stride = 2; d.out_offset = 0; d.split = 2; d.act2 = ACT_SIGMOID; d.out2 = weight;
    GS_TRY(goslam_conv2d_nhwc(&d, N, h, w, stream));
  }
  GS_TRY(goslam_nhwc_to_nchw_f16(ws.state, net_out, N, 128, hw, stream));
  if (!frame_slot) return GOSLAM_OK;
  // ---- GraphAgg (src/droid_net.py:51-67)
  GS_TRY(layer(ws.state, 128, 0, 128, W->agg1_w, W->agg1_b, 9, 128, 128, ACT_RELU, 1.f, ws.a1, 0, 128, N, h, w, stream));
  {
    const size_t total = (size_t)M * hw * 16;
    scatter_mean_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ws.a1, frame_slot, ws.mean, N, M, hw);
    GS_CHECK_LAUNCH();
  }
  GS_TRY(layer(ws.mean, 128, 0, 128, W->agg2_w, W->agg2_b, 9, 128, 128, ACT_RELU, 1.f, ws.a2, 0, 128, M, h, w, stream));
  GS_TRY(layer(ws.a2, 128, 0, 128, W->eta_w, W->eta_b, 9, 1, 16, ACT_SOFTPLUS, 0.01f, eta, 1, 1, M, h, w, stream));
  GS_TRY(layer(ws.a2, 128, 0, 128, W->upmask_w, W->upmask_b, 1, 576, 576, ACT_NONE, 1.f, ws.up, 0, 576, M, h, w, stream));
  GS_TRY(goslam_nhwc_to_nchw_f16(ws.up, upmask, M, 576, hw, stream));
#undef GS_TRY
  return GOSLAM_OK;
}

int goslam_conv_gru(const goslam_gru_weights* wts, const void* net, const void* inp, const void* corr,
                    const void* flow, void* net_out, int B, int h, int w, void* workspace,
                    size_t workspace_bytes, void* stream) {
  if (!wts || B < 0 || h <= 0 || w <= 0) return GOSLAM_EINVAL;
  if (B == 0) return GOSLAM_OK;
  GruWs ws;
  const size_t need = gru_layout(B, h, w, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  ConvMaps m{};
  ConvParams p{};
  p.B = B; p.h = h; p.w = w;
  p.net = reinterpret_cast<const __half*>(net);
  // ---- pass G: glo_sum = sum_px sigmoid(w(net)) * net
  if (!act_map(net, B, h, w, 128, &m.in[0]) || !weight_map(wts->w_w, 1, 128, 128, &m.w)) return GOSLAM_ELAUNCH;
  p.n_nt = 1;
  p.taps = 1; p.n_in = 1; p.chunks[0] = 2; p.N = 128; p.epi = EPI_GLO; p.bias = wts->b_w; p.glo = nullptr;
  p.glo_sum = ws.glo_sum;
  int rc = conv_launch(m, p, st);
  if (rc) return rc;
  gru_glo_fc_kernel<<<B, 256, 0, st>>>(ws.glo_sum, gs_cdiv(h, kPY) * gs_cdiv(w, kPX) * 4, wts->w_glo, wts->b_glo, ws.glo,
                                       1.0f / (float)(h * w));
  GS_CHECK_LAUNCH();
  // ---- pass ZR: z, r*net
  if (!act_map(inp, B, h, w, 128, &m.in[1]) || !act_map(corr, B, h, w, 128, &m.in[2]) ||
      !act_map(flow, B, h, w, 64, &m.in[3]) || !weight_map(wts->w_zr, 9, 256, 448, &m.w))
    return GOSLAM_ELAUNCH;
  p.taps = 9; p.n_in = 4; p.chunks[0] = 2; p.chunks[1] = 2; p.chunks[2] = 2; p.chunks[3] = 1;
  p.N = 256; p.epi = EPI_ZR; p.bias = wts->b_zr; p.glo = ws.glo; p.z_out = ws.z; p.rnet_out = ws.rnet;
  rc = conv_launch(m, p, st);
  if (rc) return rc;
  // ---- pass Q: net' = (1 - z) net + z tanh(convq([r*net | inp | corr | flow]) + glo_q)
  if (!act_map(ws.rnet, B, h, w, 128, &m.in[0]) || !weight_map(wts->w_q, 9, 128, 448, &m.w)) return GOSLAM_ELAUNCH;
  p.N = 128; p.epi = EPI_Q; p.bias = wts->b_q; p.z_in = ws.z; p.net_out = reinterpret_cast<__half*>(net_out);
  return conv_launch(m, p, st);
}

}  // extern "C"
