// neus.cu — fused hash-grid neural-surface ray marcher (InstantNeuS.forward).
//
// Replaces, in ONE persistent kernel: tiny-cuda-nn HashGrid forward + its input-gradient
// backward (SDF normal), nn.Linear(35,32), NeuS alpha, sin-embedding, tiny-cuda-nn
// FullyFusedMLP 67(->80)->64->64->3(->16), sigmoid, and front-to-back compositing
// (src/InstantNeuS.py:295-370 with :12-32, :35-94, :97-160, :162-205, :258-293), i.e. what
// the reference runs as ~60 eager kernels + two tcnn launches + an autograd pass.
//
// tiny-cuda-nn is an un-vendored, un-pinned dependency of the reference (README.md:95); its
// arithmetic is restated from its published algorithm (see oracle/neus_oracle.py header):
//   * level l: scale = exp2(l*log2(b))*16 - 1, res = ceil(scale)+1, pos = x*scale + 0.5,
//     8-corner trilinear; index = x + y*res + z*res^2 while the stride fits the table,
//     else (x*1) ^ (y*2654435761) ^ (z*805459861); mod table size; table entries half2;
//     features accumulated in half:  r += (half)(w * (float)v);
//   * d(enc)/dx in fp32 from half table values, dL/dy rounded to half (tcnn backward);
//   * MLP: half inputs padded with 1.0 to 80, half activations, ReLU, no bias; we accumulate
//     in fp32 on mma.sync (tcnn: half accumulators) — documented tolerance in the tests.
//
// Work decomposition: a block owns kRaysPerGroup rays at a time (persistent loop).  A warp
// takes 32 consecutive samples: phase 1 is one thread per sample (gather + SDF head +
// alpha + embedding), phase 2 is the warp-wide MLP on m16n8k16 tensor-core tiles with the
// weights resident in shared memory, phase 3 composites each ray with a warp scan.
#include "common.cuh"
#include "launch.cuh"
#include <math.h>
#include <algorithm>

namespace {

constexpr int kLevels = 16;
// code-size knobs (the kernel body is ~60 KB of SASS; ncu shows warps starved on instruction fetch)
constexpr int kNeusKUnroll = 8, kNeusHUnroll = 1;
constexpr int kThreadsN = 384;
constexpr int kWarpsN = kThreadsN / 32;
constexpr int kDenseLevels = 5;     // levels whose res^3 fits the table (16,24,34,49,71)
constexpr int kIn = 80, kInPad = 88;     // MLP input width / padded smem row (halves)
constexpr int kHid = 64, kHidPad = 72;
constexpr int kOutW = 16;

struct GridMeta {
  float scale[kLevels];
  int res[kLevels];
  unsigned offset[kLevels];   // in entries (half2)
  unsigned size[kLevels];     // entries in level
};

GridMeta make_grid_meta(int64_t* total_entries) {
  GridMeta g{};
  const float log2_b = log2f(1.447269237440378f);
  unsigned off = 0;
  for (int l = 0; l < kLevels; ++l) {
    const float scale = exp2f((float)l * log2_b) * 16.0f - 1.0f;
    const unsigned res = (unsigned)ceilf(scale) + 1u;
    unsigned long long dense = (unsigned long long)res * res * res;
    const unsigned long long maxp = 0xFFFFFFFFull / 2;
    unsigned long long p = dense > maxp ? maxp : dense;
    p = (p + 7) / 8 * 8;
    if (p > (1ull << 19)) p = 1ull << 19;
    g.scale[l] = scale; g.res[l] = (int)res; g.offset[l] = off; g.size[l] = (unsigned)p;
    off += (unsigned)p;
  }
  if (total_entries) *total_entries = off;
  return g;
}


struct NeusArgs {
  goslam_neus_params p;
  goslam_neus_out o;
  const float* rays_o; const float* rays_d; const float* z_vals; const float* dists;
  int R, S;
  float* blk_gerr;        // [grid] partial sums of the eikonal term
  unsigned* blk_count;    // [grid] in-bound sample counts
  int* flag;              // [1] written by the finalize kernel: 1 = nothing in bound
  int mode;               // 0 main pass, 1 fix-up pass (mask[:100] = True)
  int rays_per_group;     // rays one warp composites together (rays_per_group * S <= kMaxGroup)
};

__device__ __forceinline__ void ldmatrix_x4(unsigned (&r)[4], const void* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldmatrix_x2(unsigned (&r)[2], const void* p) {
  const unsigned a = (unsigned)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n"
               : "=r"(r[0]), "=r"(r[1]) : "r"(a));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const unsigned (&a)[4],
                                         const unsigned (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// One dense layer for a 32-row warp tile: out[32][N] = in[32][K] * W[N][K]^T (fp32 accum).
// NT = N/8 n-tiles, KT = K/16 k-steps.  acc[mt][nt][4].
template <int NT, int KT, int IN_LD, int W_LD>
__device__ __forceinline__ void warp_layer(const __half* in, const __half* W,
                                           float (&acc)[2][NT][4], int lane) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[mt][nt][q] = 0.f;
  const int lr = lane & 15, lc = (lane >> 4) * 8;       // ldmatrix.x4 A addressing
  const int br = lane & 7, bc = ((lane >> 3) & 1) * 8;  // ldmatrix.x2 B addressing
#pragma unroll kNeusKUnroll
  for (int kt = 0; kt < KT; ++kt) {
    unsigned a[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
      ldmatrix_x4(a[mt], in + (mt * 16 + lr) * IN_LD + kt * 16 + lc);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      unsigned b[2];
      ldmatrix_x2(b, W + (nt * 8 + br) * W_LD + kt * 16 + bc);
      mma16816(acc[0][nt], a[0], b);
      mma16816(acc[1][nt], a[1], b);
    }
  }
}

template <int NT, int OUT_LD>
__device__ __forceinline__ void store_relu_half(const float (&acc)[2][NT][4], __half* out,
                                                int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int col = nt * 8 + 2 * t;
      const __half2 lo = __floats2half2_rn(fmaxf(acc[mt][nt][0], 0.f), fmaxf(acc[mt][nt][1], 0.f));
      const __half2 hi = __floats2half2_rn(fmaxf(acc[mt][nt][2], 0.f), fmaxf(acc[mt][nt][3], 0.f));
      *reinterpret_cast<__half2*>(out + (mt * 16 + g) * OUT_LD + col) = lo;
      *reinterpret_cast<__half2*>(out + (mt * 16 + g + 8) * OUT_LD + col) = hi;
    }
}

// ---------------------------------------------------------------------------------------
// Shared memory: network weights once per (persistent) block + a private slab per warp.
// ---------------------------------------------------------------------------------------
constexpr int kEncPad = 40;            // enc row stride (halves): 80 B, conflict-free ldmatrix
constexpr int kMaxGroup = 288;         // samples per warp work item (rays_per_group * S): 4 rays x 72

struct WarpSlab {
  alignas(16) __half actA[32 * kInPad];    // MLP input rows / hidden 2; also the fp32 SDF-head tile
  alignas(16) __half actB[32 * kHidPad];   // enc rows (stride kEncPad) then hidden 1, rgb scratch
  float w[kMaxGroup];                      // compositing weights of the open group
};
// Shared memory is sized so that 12 warps + the weights stay under the 164 KB carve-out step:
// the remaining ~90 KB of the SM's 256 KB serve as L1 for the hash-grid gathers (measured:
// 14 warps with a 228 KB carve-out are 40 % SLOWER than 12 warps, 8 warps with 124 KB L1 only
// 3 % slower).  Mid-point depths for the variance pass are recomputed from z_vals/dists.

struct Smem {
  alignas(16) __half W1[kHid * kInPad];
  alignas(16) __half W2[kHid * kHidPad];
  alignas(16) __half W3[kOutW * kHidPad];
  alignas(16) __half sdfWhi[32 * kEncPad];   // Linear(35,32) weight, enc part, fp16 hi/lo split:
  alignas(16) __half sdfWlo[32 * kEncPad];   //   W = hi + lo to 2^-22 relative, products exact
  alignas(16) float sdfWxyz[3 * 32];         // xyz part [k][out], fp32
  alignas(16) float sdfB[32];
  float gy[32];                              // dL/dy of the normal: W[0,3:] rounded to half
  float colB[3 * 33];
  WarpSlab slab[kWarpsN];
  float red_g[kWarpsN];
  unsigned red_c[kWarpsN];
};

static_assert(32 * 33 * 4 <= 32 * kInPad * 2, "fp32 SDF-head tile must fit in actA");
static_assert(kThreadsN != 384 || sizeof(Smem) + 1024 <= 164 * 1024, "12-warp layout must fit the 164 KB carve-out");

struct LevelConst {
  float scale;
  unsigned res, res2, offset, size;
};
__constant__ LevelConst c_lvl[kLevels];

// sin(x) for |x| up to a few hundred: 2-term Cody-Waite reduction by 2*pi, then the SFU.
__device__ __forceinline__ float fast_sin(float x) {
  // rint via the 1.5*2^23 magic constant (exact for |v| < 2^22; the conversion unit is quarter rate)
  const float k = __fsub_rn(__fadd_rn(x * 0.15915494309189535f, 12582912.0f), 12582912.0f);
  float r = fmaf(-k, 6.28125f, x);
  r = fmaf(-k, 1.9353071795864769e-3f, r);
  return __sinf(r);
}

__device__ __forceinline__ unsigned h2_as_u32(__half2 h) { return *reinterpret_cast<unsigned*>(&h); }

__device__ __forceinline__ void encode_level(int l, const bool HASHED, const __half2* __restrict__ table,
                                             const float (&x01)[3], const float* gyv,
                                             __half2& enc, float (&genc)[3]) {
  const LevelConst L = c_lvl[l];
  float fr[3];
  unsigned pg[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float pos = fmaf(L.scale, x01[c], 0.5f);
    // floor of a float in [0, 2^23) without the quarter-rate conversion unit: adding 2^23 with
    // round-toward-zero drops the fraction, the integer is then the low mantissa bits (exact)
    const float t = __fadd_rz(pos, 8388608.0f);
    const float fl = t - 8388608.0f;
    pg[c] = __float_as_uint(t) & 0x7FFFFFu;
    fr[c] = pos - fl;
  }
  unsigned idx[8];
  if (HASHED) {
    // (a ^ b ^ c) & m == (a & m) ^ (b & m) ^ (c & m): mask the six components once, one LOP3 per corner
    const unsigned hx0 = pg[0] & 0x7FFFFu, hx1 = (pg[0] + 1u) & 0x7FFFFu;
    const unsigned hy = pg[1] * 2654435761u, hz = pg[2] * 805459861u;
    const unsigned hy0 = hy & 0x7FFFFu, hy1 = (hy + 2654435761u) & 0x7FFFFu;
    const unsigned hz0 = hz & 0x7FFFFu, hz1 = (hz + 805459861u) & 0x7FFFFu;
#pragma unroll
    for (int q = 0; q < 8; ++q)
      idx[q] = ((q & 1) ? hx1 : hx0) ^ ((q & 2) ? hy1 : hy0) ^ ((q & 4) ? hz1 : hz0);
  } else {
    // dense level: tcnn's `index % size`.  pos = x*scale + 0.5 reaches res-1+0.5, so the +1
    // corner can index one past the last row/plane and wraps; index < 2*size always, so the
    // modulo is one conditional subtract.
    const unsigned base = pg[0] + pg[1] * L.res + pg[2] * L.res2;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const unsigned i = base + ((q & 1) ? 1u : 0u) + ((q & 2) ? L.res : 0u) + ((q & 4) ? L.res2 : 0u);
      idx[q] = i >= L.size ? i - L.size : i;
    }
  }
  // level base as an integer so that each gather address is ONE wide multiply-add (idx * 4 + base)
  const unsigned long long lvl = reinterpret_cast<unsigned long long>(table) + (unsigned long long)L.offset * 4ull;
  __half2 v[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    unsigned long long addr;
    asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(addr) : "r"(idx[q]), "l"(lvl));
    v[q] = __ldg(reinterpret_cast<const __half2*>(addr));
  }

  const float wx[2] = {1.f - fr[0], fr[0]}, wy[2] = {1.f - fr[1], fr[1]}, wz[2] = {1.f - fr[2], fr[2]};
  __half2 r = __float2half2_rn(0.f);
  float2 vf[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    vf[q] = __half22float2(v[q]);
    const float w = (wx[q & 1] * wy[(q >> 1) & 1]) * wz[(q >> 2) & 1];
    r = __hadd2_rn(r, __floats2half2_rn(w * vf[q].x, w * vf[q].y));      // half accumulation (tcnn)
  }
  enc = r;
  // d(sdf)/d(x01) through this level: contract the two features with dL/dy first (c = v . gy at
  // the 8 corners), then the gradient of the trilinear interpolant of that one scalar field.
  const float gy0 = gyv[2 * l], gy1 = gyv[2 * l + 1];
  float c[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) c[q] = fmaf(vf[q].y, gy1, vf[q].x * gy0);
  const float dx0 = c[1] - c[0], dx1 = c[3] - c[2], dx2 = c[5] - c[4], dx3 = c[7] - c[6];
  const float dy0 = c[2] - c[0], dy1 = c[3] - c[1], dy2 = c[6] - c[4], dy3 = c[7] - c[5];
  const float dz0 = c[4] - c[0], dz1 = c[5] - c[1], dz2 = c[6] - c[2], dz3 = c[7] - c[3];
  const float gx = wz[0] * fmaf(wy[1], dx1, wy[0] * dx0) + wz[1] * fmaf(wy[1], dx3, wy[0] * dx2);
  const float gyy = wz[0] * fmaf(wx[1], dy1, wx[0] * dy0) + wz[1] * fmaf(wx[1], dy3, wx[0] * dy2);
  const float gz = wy[0] * fmaf(wx[1], dz1, wx[0] * dz0) + wy[1] * fmaf(wx[1], dz3, wx[0] * dz2);
  genc[0] = fmaf(L.scale, gx, genc[0]);
  genc[1] = fmaf(L.scale, gyy, genc[1]);
  genc[2] = fmaf(L.scale, gz, genc[2]);
}

__global__ void __launch_bounds__(kThreadsN, 1)
neus_forward_kernel(const NeusArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int S = a.S;
  const int G = a.rays_per_group;                 // rays per warp work item
  const int gs = G * S;                           // real samples per item (<= kMaxGroup)
  const int ntiles = gs_cdiv_dev(gs, 32);

  int num_groups = gs_cdiv_dev(a.R, G);
  if (a.mode == 1) {
    if (*a.flag == 0) return;                     // something was in bound: no fix-up needed
    const int need = gs_cdiv_dev(gs_cdiv_dev(100, S), G);
    if (num_groups > need) num_groups = need;
  }

  // ---- stage the network weights once per block (persistent) ----
  {
    const __half* w = reinterpret_cast<const __half*>(a.p.mlp_w);
    for (int i = tid; i < kHid * kIn; i += kThreadsN) sm.W1[(i / kIn) * kInPad + i % kIn] = w[i];
    for (int i = tid; i < kHid * kHid; i += kThreadsN)
      sm.W2[(i / kHid) * kHidPad + i % kHid] = w[kHid * kIn + i];
    for (int i = tid; i < kOutW * kHid; i += kThreadsN)
      sm.W3[(i / kHid) * kHidPad + i % kHid] = w[kHid * kIn + kHid * kHid + i];
    for (int i = tid; i < 32 * 35; i += kThreadsN) {
      const int o = i / 35, k = i % 35;
      const float wv = a.p.sdf_w[i];
      if (k < 3) {
        sm.sdfWxyz[k * 32 + o] = wv;
      } else {
        const __half hi = __float2half_rn(wv);
        sm.sdfWhi[o * kEncPad + (k - 3)] = hi;
        sm.sdfWlo[o * kEncPad + (k - 3)] = __float2half_rn(wv - __half2float(hi));
        if (o == 0) sm.gy[k - 3] = __half2float(hi);
      }
    }
    for (int i = tid; i < 32 * (kEncPad - 32); i += kThreadsN) {   // zero the row padding
      const int o = i / (kEncPad - 32), k = 32 + i % (kEncPad - 32);
      sm.sdfWhi[o * kEncPad + k] = __float2half_rn(0.f);
      sm.sdfWlo[o * kEncPad + k] = __float2half_rn(0.f);
    }
    for (int i = tid; i < 32; i += kThreadsN) sm.sdfB[i] = a.p.sdf_b[i];
    for (int i = tid; i < 99; i += kThreadsN) sm.colB[i] = a.p.color_B[i];
  }
  __syncthreads();

  WarpSlab& sl = sm.slab[warp];
  const __half2* table = reinterpret_cast<const __half2*>(a.p.grid);
  float gerr_local = 0.f;
  unsigned count_local = 0;
  const int warps_total = gridDim.x * kWarpsN;

  for (int group = blockIdx.x * kWarpsN + warp; group < num_groups; group += warps_total) {
    const int ray0 = group * G;
    const int nrays = min(G, a.R - ray0);
    const int nsamp = nrays * S;

    // compositing state of the ray that is still open (lane-replicated)
    int open_ray = -1;
    float carry_T = 1.f;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // ws, dep, r, g, b, nx, ny, nz

    for (int tile = 0; tile < ntiles; ++tile) {
      if (tile * 32 >= nsamp) break;               // warp-uniform
      const int ls = tile * 32 + lane;             // local sample index in the group
      const bool valid = ls < nsamp;
      const int lr = valid ? ls / S : -2;          // local ray
      const int sidx = valid ? ls - lr * S : 0;
      const int ray = ray0 + (valid ? lr : 0);
      const size_t gidx = (size_t)ray * S + sidx;

      float zm = 0.f, dist = 0.f, alpha = 0.f, sdf = 100.f;
      float g3[3] = {0.f, 0.f, 0.f}, dir[3] = {0.f, 0.f, 0.f}, pt[3] = {0.f, 0.f, 0.f};
      float xn[3] = {0.f, 0.f, 0.f}, dscale[3] = {0.f, 0.f, 0.f};
      bool inb = false;
      if (valid) {
        dist = a.dists[gidx];
        zm = __fadd_rn(a.z_vals[gidx], dist / 2.0f);
        // op-by-op fp32 like the reference's separate torch kernels (no FMA contraction): the
        // hash grid turns a 1-ulp difference in the position into a different fine-level cell
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          dir[c] = a.rays_d[(size_t)ray * 3 + c];
          pt[c] = __fadd_rn(a.rays_o[(size_t)ray * 3 + c], __fmul_rn(dir[c], zm));
        }
        inb = pt[0] < a.p.rt_bound[1] && pt[0] > a.p.rt_bound[0] &&
              pt[1] < a.p.rt_bound[3] && pt[1] > a.p.rt_bound[2] &&
              pt[2] < a.p.rt_bound[5] && pt[2] > a.p.rt_bound[4];
        if (a.mode == 1 && gidx < 100) inb = true;
      }

      // ---- phase 1a: hash-grid encoding (thread per sample) -> enc row in actB ----
      float genc[3] = {0.f, 0.f, 0.f};
      __half2* encrow = reinterpret_cast<__half2*>(sl.actB + lane * kEncPad);
      if (inb) {
        float x01[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float b0 = a.p.bound[2 * c], b1 = a.p.bound[2 * c + 1];
          const float raw = __fsub_rn(__fmul_rn(__fdiv_rn(__fsub_rn(pt[c], b0), __fsub_rn(b1, b0)), 2.0f), 1.0f);
          xn[c] = fminf(fmaxf(raw, -1.0f), 1.0f);
          dscale[c] = (raw >= -1.0f && raw <= 1.0f) ? 2.0f / (b1 - b0) : 0.0f;
          x01[c] = __fdiv_rn(__fadd_rn(xn[c], 1.0f), 2.0f);
        }
#pragma unroll kNeusHUnroll
        for (int l = 0; l < kLevels; ++l) {                 // one copy of the gather/interpolation code
          __half2 e;
          encode_level(l, l >= kDenseLevels, table, x01, sm.gy, e, genc);
          encrow[l] = e;
        }
      } else {
#pragma unroll
        for (int l = 0; l < kLevels; ++l) encrow[l] = __float2half2_rn(0.f);
      }
      if (a.o.enc && valid) {                        // training pass: keep the encoding row (64 B)
        uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(a.o.enc) + gidx * 32);
        const uint4* src = reinterpret_cast<const uint4*>(encrow);
#pragma unroll
        for (int v = 0; v < 4; ++v) dst[v] = src[v];
      }
      __syncwarp();

      // ---- phase 1b: SDF head  out[32 x 32] = enc (W_hi + W_lo)^T  on tensor cores ----
      float* outf = reinterpret_cast<float*>(sl.actA);     // [32][33] fp32 tile
      {
        float acc4[2][4][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc4[mt][nt][q] = 0.f;
        const int lrr = lane & 15, lcc = (lane >> 4) * 8;
        const int br = lane & 7, bc = ((lane >> 3) & 1) * 8;
#pragma unroll
        for (int kt = 0; kt < 2; ++kt) {
          unsigned af[2][4];
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
            ldmatrix_x4(af[mt], sl.actB + (mt * 16 + lrr) * kEncPad + kt * 16 + lcc);
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) {
            unsigned bh[2], bl[2];
            ldmatrix_x2(bh, sm.sdfWhi + (nt * 8 + br) * kEncPad + kt * 16 + bc);
            ldmatrix_x2(bl, sm.sdfWlo + (nt * 8 + br) * kEncPad + kt * 16 + bc);
            mma16816(acc4[0][nt], af[0], bl);
            mma16816(acc4[1][nt], af[1], bl);
            mma16816(acc4[0][nt], af[0], bh);
            mma16816(acc4[1][nt], af[1], bh);
          }
        }
        const int g = lane >> 2, t = lane & 3;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) {
            const int col = nt * 8 + 2 * t;
            outf[(mt * 16 + g) * 33 + col] = acc4[mt][nt][0];
            outf[(mt * 16 + g) * 33 + col + 1] = acc4[mt][nt][1];
            outf[(mt * 16 + g + 8) * 33 + col] = acc4[mt][nt][2];
            outf[(mt * 16 + g + 8) * 33 + col + 1] = acc4[mt][nt][3];
          }
      }
      __syncwarp();
      float out[32];
#pragma unroll
      for (int o4 = 0; o4 < 8; ++o4) {
        const float4 bb = reinterpret_cast<const float4*>(sm.sdfB)[o4];
        const float4 w0 = reinterpret_cast<const float4*>(sm.sdfWxyz)[o4];
        const float4 w1 = reinterpret_cast<const float4*>(sm.sdfWxyz + 32)[o4];
        const float4 w2 = reinterpret_cast<const float4*>(sm.sdfWxyz + 64)[o4];
        const float* of = outf + lane * 33 + 4 * o4;
        out[4 * o4 + 0] = of[0] + (bb.x + w0.x * xn[0] + w1.x * xn[1] + w2.x * xn[2]);
        out[4 * o4 + 1] = of[1] + (bb.y + w0.y * xn[0] + w1.y * xn[1] + w2.y * xn[2]);
        out[4 * o4 + 2] = of[2] + (bb.z + w0.z * xn[0] + w1.z * xn[1] + w2.z * xn[2]);
        out[4 * o4 + 3] = of[3] + (bb.w + w0.w * xn[0] + w1.w * xn[1] + w2.w * xn[2]);
      }
      __syncwarp();                                  // everyone has read outf before actA is reused

      if (inb) {
        sdf = out[0];
#pragma unroll
        for (int c = 0; c < 3; ++c) g3[c] = (sm.sdfWxyz[c * 32] + 0.5f * genc[c]) * dscale[c];
      }

      // ---- NeuS alpha (get_alpha, src/InstantNeuS.py:276-293) ----
      if (valid) {
        const float true_cos = dir[0] * g3[0] + dir[1] * g3[1] + dir[2] * g3[2];
        const float car = a.p.cos_anneal_ratio;
        const float iter_cos = -(fmaxf(-true_cos * 0.5f + 0.5f, 0.f) * (1.0f - car) +
                                 fmaxf(-true_cos, 0.f) * car);
        const float half_step = iter_cos * dist / 2.0f;
        const float prev_cdf = 1.0f / (1.0f + expf(-(sdf - half_step) * a.p.inv_s));
        const float next_cdf = 1.0f / (1.0f + expf(-(sdf + half_step) * a.p.inv_s));
        alpha = (prev_cdf - next_cdf + 1e-5f) / (prev_cdf + 1e-5f);
        alpha = fminf(fmaxf(alpha, 0.f), 1.f);
        alpha = inb ? alpha : 0.f;
        a.o.sdf[gidx] = sdf;
        a.o.z_mid[gidx] = zm;
        if (a.o.alpha) a.o.alpha[gidx] = alpha;
        if (a.o.grad) {
#pragma unroll
          for (int c = 0; c < 3; ++c) a.o.grad[gidx * 3 + c] = g3[c];
        }
        if (a.o.pos) {
#pragma unroll
          for (int c = 0; c < 3; ++c) a.o.pos[gidx * 3 + c] = xn[c];
        }
        if (inb) {
          const float gn = sqrtf(g3[0] * g3[0] + g3[1] * g3[1] + g3[2] * g3[2]) - 1.0f;
          gerr_local += gn * gn;
          ++count_local;
        }
      }

      // ---- MLP input row: [sin(p B)(33) | normal(3) | feat(31) | 1-padding(13)] ----
      {
        // the first 32 embedding columns in a rolled loop (4 per trip: the kernel is instruction-
        // fetch sensitive, see kNeusHUnroll), column 32 with the static tail of the row
        __half* rowh = sl.actA + lane * kInPad;                            // 176-byte rows: 16-B aligned
#pragma unroll 1
        for (int j4 = 0; j4 < 8; ++j4) {
          float sn[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int j = 4 * j4 + u;
            sn[u] = fast_sin(pt[0] * sm.colB[j] + pt[1] * sm.colB[33 + j] + pt[2] * sm.colB[66 + j]);
          }
          *reinterpret_cast<uint2*>(rowh + 4 * j4) =
              make_uint2(h2_as_u32(__floats2half2_rn(sn[0], sn[1])), h2_as_u32(__floats2half2_rn(sn[2], sn[3])));
        }
        float row[kIn - 32];                                               // columns 32 .. 79
        row[0] = fast_sin(pt[0] * sm.colB[32] + pt[1] * sm.colB[65] + pt[2] * sm.colB[98]);
#pragma unroll
        for (int c = 0; c < 3; ++c) row[1 + c] = g3[c];
#pragma unroll
        for (int i = 0; i < 31; ++i) row[4 + i] = inb ? out[1 + i] : 0.f;
#pragma unroll
        for (int i = 35; i < kIn - 32; ++i) row[i] = 1.0f;
        uint4* rowA = reinterpret_cast<uint4*>(rowh + 32);
#pragma unroll
        for (int v8 = 0; v8 < (kIn - 32) / 8; ++v8) {
          uint4 u;
          u.x = h2_as_u32(__floats2half2_rn(row[8 * v8 + 0], row[8 * v8 + 1]));
          u.y = h2_as_u32(__floats2half2_rn(row[8 * v8 + 2], row[8 * v8 + 3]));
          u.z = h2_as_u32(__floats2half2_rn(row[8 * v8 + 4], row[8 * v8 + 5]));
          u.w = h2_as_u32(__floats2half2_rn(row[8 * v8 + 6], row[8 * v8 + 7]));
          rowA[v8] = u;
        }
        if (a.o.mlp_in && valid) {                   // training pass: keep the MLP input row (160 B)
          uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(a.o.mlp_in) + gidx * kIn);
          const uint4* src = reinterpret_cast<const uint4*>(rowh);
#pragma unroll
          for (int v = 0; v < kIn / 8; ++v) dst[v] = src[v];
        }
      }
      __syncwarp();

      // ---- warp-wide MLP on tensor cores ----
      float rgbv[3] = {0.f, 0.f, 0.f};
      {
        float accm[2][8][4];
        warp_layer<8, kIn / 16, kInPad, kInPad>(sl.actA, sm.W1, accm, lane);
        store_relu_half<8, kHidPad>(accm, sl.actB, lane);
        __syncwarp();
        warp_layer<8, kHid / 16, kHidPad, kHidPad>(sl.actB, sm.W2, accm, lane);
        __syncwarp();
        store_relu_half<8, kInPad>(accm, sl.actA, lane);
        __syncwarp();
        float acc3[2][2][4];
        warp_layer<2, kHid / 16, kInPad, kHidPad>(sl.actA, sm.W3, acc3, lane);
        __syncwarp();
        float* scratch = reinterpret_cast<float*>(sl.actB);   // 32 x 4 floats
        const int g = lane >> 2, t = lane & 3;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          if (t < 2) {
            scratch[(mt * 16 + g) * 4 + 2 * t] = acc3[mt][0][0];
            scratch[(mt * 16 + g) * 4 + 2 * t + 1] = acc3[mt][0][1];
            scratch[(mt * 16 + g + 8) * 4 + 2 * t] = acc3[mt][0][2];
            scratch[(mt * 16 + g + 8) * 4 + 2 * t + 1] = acc3[mt][0][3];
          }
        }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float x = __half2float(__float2half_rn(scratch[lane * 4 + c]));   // tcnn output is half
          const float sg = 1.0f / (1.0f + expf(-x));
          rgbv[c] = inb ? __half2float(__float2half_rn(sg)) : 0.f;                // torch.sigmoid(half)
          if (a.o.rgb && valid) a.o.rgb[gidx * 3 + c] = rgbv[c];
        }
        __syncwarp();
      }

      // ---- incremental front-to-back compositing (segmented scan over the rays in this tile) ----
      {
        const float fct = valid ? (1.0f - alpha + 1e-7f) : 1.0f;
        float inc = fct;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const float nb = __shfl_up_sync(0xffffffffu, inc, off);
          const int nr = __shfl_up_sync(0xffffffffu, lr, off);
          if (lane >= off && nr == lr) inc *= nb;
        }
        float exc = __shfl_up_sync(0xffffffffu, inc, 1);
        const int prev_lr = __shfl_up_sync(0xffffffffu, lr, 1);
        if (lane == 0 || prev_lr != lr) exc = 1.0f;
        const float T = (lr == open_ray ? carry_T : 1.0f) * exc;
        const float wgt = alpha * T;
        if (valid) sl.w[ls] = wgt;
        const int first_ray = (tile * 32) / S;
        const int last_ray = min((tile * 32 + 31) / S, nrays - 1);
        // carry for the ray that stays open after this tile
        const int last_lane = min(31, nsamp - 1 - tile * 32);
        const float inc_last = __shfl_sync(0xffffffffu, inc, last_lane);
        const float carry_next = (last_ray == open_ray ? carry_T : 1.0f) * inc_last;
        for (int q = first_ray; q <= last_ray; ++q) {
          const bool mine = valid && lr == q;
          float v8[8];
          v8[0] = mine ? wgt : 0.f;
          v8[1] = mine ? zm * wgt : 0.f;
          v8[2] = mine ? rgbv[0] * wgt : 0.f;
          v8[3] = mine ? rgbv[1] * wgt : 0.f;
          v8[4] = mine ? rgbv[2] * wgt : 0.f;
          const float m = inb ? 1.f : 0.f;
          v8[5] = mine ? g3[0] * wgt * m : 0.f;
          v8[6] = mine ? g3[1] * wgt * m : 0.f;
          v8[7] = mine ? g3[2] * wgt * m : 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) v8[i] = gs_warp_sum(v8[i]) + (q == open_ray ? acc[i] : 0.f);
          const bool done = (q + 1) * S <= tile * 32 + 32;      // last sample of ray q is in this tile
          if (done) {
            const float dep = v8[1];
            float var = 0.f;
            __syncwarp();
            for (int s = lane; s < S; s += 32) {
              const size_t gi = (size_t)(ray0 + q) * S + s;
              const float dz = __fadd_rn(a.z_vals[gi], a.dists[gi] / 2.0f) - dep;
              var += dz * dz * sl.w[q * S + s];
            }
            var = gs_warp_sum(var);
            if (lane == 0) {
              const int rg = ray0 + q;
              a.o.weight_sum[rg] = v8[0]; a.o.depth[rg] = dep; a.o.depth_variance[rg] = var;
              a.o.color[(size_t)rg * 3 + 0] = v8[2]; a.o.color[(size_t)rg * 3 + 1] = v8[3];
              a.o.color[(size_t)rg * 3 + 2] = v8[4];
              a.o.normal[(size_t)rg * 3 + 0] = v8[5]; a.o.normal[(size_t)rg * 3 + 1] = v8[6];
              a.o.normal[(size_t)rg * 3 + 2] = v8[7];
            }
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[i] = v8[i];
          }
        }
        open_ray = last_ray;
        carry_T = carry_next;
        __syncwarp();
      }
    }
  }

  // ---- per-block partials of the eikonal term / in-bound count (deterministic order) ----
  gerr_local = gs_warp_sum(gerr_local);
  unsigned cnt = count_local;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) { sm.red_g[warp] = gerr_local; sm.red_c[warp] = cnt; }
  __syncthreads();
  if (tid == 0) {
    float g = 0.f; unsigned c = 0;
    for (int w = 0; w < kWarpsN; ++w) { g += sm.red_g[w]; c += sm.red_c[w]; }
    a.blk_gerr[blockIdx.x] = g;
    a.blk_count[blockIdx.x] = c;
  }
}

__global__ void neus_finalize_kernel(const float* blk_gerr, const unsigned* blk_count, int nblk,
                                     long long total_samples, float* gradient_error, int* flag,
                                     int mode) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (mode == 1 && *flag == 0) return;
  double g = 0.0; unsigned long long c = 0;
  for (int i = 0; i < nblk; ++i) { g += (double)blk_gerr[i]; c += blk_count[i]; }
  *gradient_error = (float)(g / (double)total_samples);
  if (mode == 0) *flag = (c == 0) ? 1 : 0;
}

// ======================================================================================================
// Renderer backward (SURVEY §8f-3: Mapper.optimize_map, src/mapping.py:60-148, differentiates
// InstantNeuS.forward, src/InstantNeuS.py:295-370, through autograd + tiny-cuda-nn).  The training pass is the SAME
// fused forward kernel with its per-sample intermediates kept (alpha, normal, sdf, rgb, MLP input row, encoding);
// the backward is two kernels around the colour network's plain GEMMs (cuBLAS through the host mirror):
//   neus_composite_bwd_kernel  dL/d{color, depth, sdf, gradient_error} -> per sample dL/d{MLP output, sdf, normal}
//                              (compositing, NeuS alpha, sigmoid, eikonal term) and dL/d(inv_s)
//   neus_grid_bwd_kernel       dL/d{encoding, normal} -> hash-grid gradient (scatter) and the part of dL/dW_sdf[0,:]
//                              that flows through the ANALYTIC normal (second order: the normal is d sdf / d x)
// ======================================================================================================
struct CompBwdArgs {
  goslam_neus_params p;
  const float* rays_o; const float* rays_d; const float* dists;
  const float* alpha; const float* rgb; const float* sdf; const float* grad; const float* z_mid;   // saved by the forward
  const float* d_color; const float* d_depth; const float* d_sdf;                                  // upstream (may be null)
  const float* d_gerr;               // dL/d gradient_error[0] (device scalar, may be null)
  float gerr_norm;                   // 1 / (number of samples gradient_error averages over)
  float* d_mlp_out;                  // [R,S,3]
  float* d_sdf_out;                  // [R,S]
  float* d_grad;                     // [R,S,3]
  float* d_inv_s;                    // [1], accumulated
  int R, S;
};

constexpr int kCompChunks = 4;       // S <= 128

// one warp per ray
__global__ void __launch_bounds__(256) neus_composite_bwd_kernel(const CompBwdArgs a) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= a.R) return;
  const int S = a.S, nch = (S + 31) >> 5;
  float dc[3] = {0.f, 0.f, 0.f}, dd = 0.f, o[3], dir[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (a.d_color) dc[c] = a.d_color[(size_t)r * 3 + c];
    o[c] = a.rays_o[(size_t)r * 3 + c];
    dir[c] = a.rays_d[(size_t)r * 3 + c];
  }
  if (a.d_depth) dd = a.d_depth[r];
  float al[kCompChunks], T[kCompChunks], G[kCompChunks], rg[kCompChunks][3];
  float carry = 1.f, total = 0.f;
#pragma unroll
  for (int c = 0; c < kCompChunks; ++c) {
    al[c] = 0.f; T[c] = 1.f; G[c] = 0.f; rg[c][0] = rg[c][1] = rg[c][2] = 0.f;
    if (c < nch) {
      const int sidx = c * 32 + lane;
      const bool valid = sidx < S;
      const size_t gi = (size_t)r * S + sidx;
      float zm = 0.f;
      if (valid) {
        al[c] = a.alpha[gi]; zm = a.z_mid[gi];
        rg[c][0] = a.rgb[gi * 3]; rg[c][1] = a.rgb[gi * 3 + 1]; rg[c][2] = a.rgb[gi * 3 + 2];
      }
      float inc = valid ? (1.0f - al[c] + 1e-7f) : 1.0f;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float nb = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc *= nb;
      }
      float exc = __shfl_up_sync(0xffffffffu, inc, 1);
      if (lane == 0) exc = 1.0f;
      T[c] = carry * exc;
      carry *= __shfl_sync(0xffffffffu, inc, 31);
      G[c] = dc[0] * rg[c][0] + dc[1] * rg[c][1] + dc[2] * rg[c][2] + dd * zm;     // dL/d weight
      total += gs_warp_sum(valid ? G[c] * al[c] * T[c] : 0.f);
    }
  }
  const float inv_s = a.p.inv_s, car = a.p.cos_anneal_ratio;
  const float eik = a.d_gerr ? __ldg(a.d_gerr) * a.gerr_norm : 0.f;
  float run = 0.f, dinv = 0.f;
#pragma unroll
  for (int c = 0; c < kCompChunks; ++c) {
    if (c < nch) {
      const int sidx = c * 32 + lane;
      const bool valid = sidx < S;
      const size_t gi = (size_t)r * S + sidx;
      const float w = al[c] * T[c];
      float incl = valid ? G[c] * w : 0.f;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float nb = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += nb;
      }
      const float chunk = __shfl_sync(0xffffffffu, incl, 31);
      const float suffix = total - (run + incl);          // sum_{k > s} G_k w_k
      run += chunk;
      if (valid) {
        const float zm = a.z_mid[gi], dist = a.dists[gi];
        float pt[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) pt[k] = __fadd_rn(o[k], __fmul_rn(dir[k], zm));
        const bool inb = pt[0] < a.p.rt_bound[1] && pt[0] > a.p.rt_bound[0] && pt[1] < a.p.rt_bound[3] &&
                         pt[1] > a.p.rt_bound[2] && pt[2] < a.p.rt_bound[5] && pt[2] > a.p.rt_bound[4];
        float dx[3] = {0.f, 0.f, 0.f}, dsdf = 0.f, dg[3] = {0.f, 0.f, 0.f};
        if (inb) {
          const float d_alpha = G[c] * T[c] - suffix / (1.0f - al[c] + 1e-7f);
#pragma unroll
          for (int k = 0; k < 3; ++k) dx[k] = dc[k] * w * rg[c][k] * (1.0f - rg[c][k]);      // through the sigmoid
          // ---- NeuS alpha (get_alpha, src/InstantNeuS.py:276-293), recomputed from the saved sdf / normal ----
          const float sdf = a.sdf[gi];
          const float g3[3] = {a.grad[gi * 3], a.grad[gi * 3 + 1], a.grad[gi * 3 + 2]};
          const float tc = dir[0] * g3[0] + dir[1] * g3[1] + dir[2] * g3[2];
          const float r0 = -tc * 0.5f + 0.5f, r1 = -tc;
          const float iter_cos = -(fmaxf(r0, 0.f) * (1.0f - car) + fmaxf(r1, 0.f) * car);
          const float hs = iter_cos * dist / 2.0f;
          const float pc = 1.0f / (1.0f + expf(-(sdf - hs) * inv_s));
          const float nc = 1.0f / (1.0f + expf(-(sdf + hs) * inv_s));
          const float araw = (pc - nc + 1e-5f) / (pc + 1e-5f);
          if (araw >= 0.f && araw <= 1.f) {                    // clip(0,1) passes the gradient inside the interval
            const float den = pc + 1e-5f;
            const float d_pc = d_alpha * (nc / (den * den));     // d/dp [(p - n + e)/(p + e)] = (n) / (p + e)^2
            const float d_nc = -d_alpha / den;
            const float d_ap = d_pc * pc * (1.0f - pc), d_an = d_nc * nc * (1.0f - nc);
            dsdf = (d_ap + d_an) * inv_s;
            const float d_hs = (d_an - d_ap) * inv_s;
            dinv += d_ap * (sdf - hs) + d_an * (sdf + hs);
            const float d_ic = d_hs * dist / 2.0f;
            const float d_tc = d_ic * ((r0 > 0.f ? 0.5f * (1.0f - car) : 0.f) + (r1 > 0.f ? car : 0.f));
#pragma unroll
            for (int k = 0; k < 3; ++k) dg[k] = d_tc * dir[k];
          }
          if (a.d_sdf) dsdf += a.d_sdf[gi];
          // ---- eikonal term: gradient_error = mean_n((|g| - 1)^2 * mask) ----
          const float gn = sqrtf(g3[0] * g3[0] + g3[1] * g3[1] + g3[2] * g3[2]);
          if (gn > 0.f) {
            const float f = eik * 2.0f * (gn - 1.0f) / gn;
#pragma unroll
            for (int k = 0; k < 3; ++k) dg[k] += f * g3[k];
          }
        }
        a.d_sdf_out[gi] = dsdf;
#pragma unroll
        for (int k = 0; k < 3; ++k) { a.d_mlp_out[gi * 3 + k] = dx[k]; a.d_grad[gi * 3 + k] = dg[k]; }
      }
    }
  }
  dinv = gs_warp_sum(dinv);
  if (lane == 0 && dinv != 0.f) atomicAdd(a.d_inv_s, dinv);
}

constexpr int kAggLevels = 8;      // levels whose scatter is reduced over runs of lanes in the same cell first
struct GridBwdArgs {
  goslam_neus_params p;
  const float* rays_o; const float* rays_d; const float* z_vals; const float* dists;
  const float* d_enc;                // [n,32]  (times *d_enc_scale when that pointer is set)
  const float* d_enc_scale;          // device scalar or null
  const float* d_grad;               // [n,3]   dL/d normal (all paths)
  float* grid_grad;                  // [entries*2], accumulated
  float* d_w0;                       // [35] dL/dW_sdf[0,:] through the normal, accumulated
  long long n; int S;
};

// thread per sample; recomputes the sample position exactly as the forward does
__global__ void __launch_bounds__(256) neus_grid_bwd_kernel(const GridBwdArgs a) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  bool act = i < a.n;
  float x01[3] = {0.f, 0.f, 0.f}, q[3] = {0.f, 0.f, 0.f}, dw_xyz[3] = {0.f, 0.f, 0.f};
  if (act) {
    const long long ray = i / a.S;
    const float dist = a.dists[i];
    const float zm = __fadd_rn(a.z_vals[i], dist / 2.0f);
    float pt[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) pt[c] = __fadd_rn(a.rays_o[ray * 3 + c], __fmul_rn(a.rays_d[ray * 3 + c], zm));
    act = pt[0] < a.p.rt_bound[1] && pt[0] > a.p.rt_bound[0] && pt[1] < a.p.rt_bound[3] && pt[1] > a.p.rt_bound[2] &&
          pt[2] < a.p.rt_bound[5] && pt[2] > a.p.rt_bound[4];
    if (act) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float b0 = a.p.bound[2 * c], b1 = a.p.bound[2 * c + 1];
        const float raw = __fsub_rn(__fmul_rn(__fdiv_rn(__fsub_rn(pt[c], b0), __fsub_rn(b1, b0)), 2.0f), 1.0f);
        const float xn = fminf(fmaxf(raw, -1.0f), 1.0f);
        const float dscale = (raw >= -1.0f && raw <= 1.0f) ? 2.0f / (b1 - b0) : 0.0f;
        x01[c] = __fdiv_rn(__fadd_rn(xn, 1.0f), 2.0f);
        const float dg = a.d_grad[i * 3 + c];
        dw_xyz[c] = dscale * dg;            // normal_c = (W0[c] + 0.5 genc_c) * dscale_c
        q[c] = 0.5f * dscale * dg;          // dL/d genc_c
      }
    }
  }
  const __half2* table = reinterpret_cast<const __half2*>(a.p.grid);
  float2* gg = reinterpret_cast<float2*>(a.grid_grad);
  const float esc = a.d_enc_scale ? 1.0f / __ldg(a.d_enc_scale) : 1.0f;
  // Two levels per trip: the 16 table gathers and the two dL/d(enc) pairs of both levels are in flight before the first
  // dependent instruction (ncu on the one-level-per-trip version: long_scoreboard 78 stalled warps per issue, no unit
  // above 35 % — latency bound).  All gathers are read-only (ld.global.nc), the scatters are fire-and-forget RED.
#pragma unroll 1
  for (int l0 = 0; l0 < kLevels; l0 += 2) {
    float fr[2][3], sc2[2];
    unsigned idx[2][8], off2[2], cell[2] = {0xffffffffu, 0xffffffffu};
    __half2 v[2][8];
    float2 de[2];
    if (act) {
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int l = l0 + u;
        const LevelConst L = c_lvl[l];
        unsigned pg[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const float pos = fmaf(L.scale, x01[c], 0.5f);
          const float fl = floorf(pos);
          pg[c] = (unsigned)fl; fr[u][c] = pos - fl;
        }
        sc2[u] = L.scale; off2[u] = L.offset;
        cell[u] = pg[0] + 4099u * pg[1] + 16785407u * pg[2];          // injective for pg < 4099 (res <= 4096)
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          const int bx = c8 & 1, by = (c8 >> 1) & 1, bz = (c8 >> 2) & 1;
          unsigned ix;
          if (l >= kDenseLevels) {
            ix = ((pg[0] + bx) ^ ((pg[1] + by) * 2654435761u) ^ ((pg[2] + bz) * 805459861u)) & 0x7FFFFu;
          } else {
            ix = (pg[0] + bx) + (pg[1] + by) * L.res + (pg[2] + bz) * L.res2;
            ix = ix >= L.size ? ix - L.size : ix;
          }
          idx[u][c8] = ix;
          v[u][c8] = __ldg(table + L.offset + ix);
        }
        de[u] = __ldg(reinterpret_cast<const float2*>(a.d_enc + i * 32 + 2 * l));
        de[u].x *= esc; de[u].y *= esc;
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int l = l0 + u;
      float t0 = 0.f, t1 = 0.f;
      // Consecutive samples of a ray sit in the same cell of the coarser levels (the 48 surface samples of a ray are ~1 cm
      // apart, a level-5 cell is 4 cm): runs of lanes with the same cell reduce their contributions with a segmented warp
      // scan and only the last lane of a run issues the 8 reductions.  Levels >= kAggLevels scatter directly.
      const bool agg = l < kAggLevels;
      unsigned run_id = 0;
      bool tail = true;
      if (agg) {                                             // warp-uniform
        const unsigned key = act ? cell[u] : 0xfffffffeu - (unsigned)lane;      // inactive lanes: runs of their own
        const unsigned prev = __shfl_up_sync(0xffffffffu, key, 1);
        const unsigned heads = __ballot_sync(0xffffffffu, lane == 0 || key != prev);
        run_id = __popc(heads & (0xffffffffu >> (31 - lane)));
        tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
      }
      float cc0[8], cc1[8];
#pragma unroll
      for (int c8 = 0; c8 < 8; ++c8) { cc0[c8] = 0.f; cc1[c8] = 0.f; }
      if (act) {
        // what the forward multiplies this level's input gradient with: dL/dy of the sdf output, rounded to half (tcnn)
        const float gy0 = __half2float(__float2half_rn(a.p.sdf_w[3 + 2 * l]));
        const float gy1 = __half2float(__float2half_rn(a.p.sdf_w[3 + 2 * l + 1]));
        const float wx[2] = {1.f - fr[u][0], fr[u][0]}, wy[2] = {1.f - fr[u][1], fr[u][1]}, wz[2] = {1.f - fr[u][2], fr[u][2]};
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          const int bx = c8 & 1, by = (c8 >> 1) & 1, bz = (c8 >> 2) & 1;
          const float w = (wx[bx] * wy[by]) * wz[bz];
          // q . grad_u(w_c): +/- the product of the other two axes' weights
          const float sdot = sc2[u] * ((bx ? q[0] : -q[0]) * (wy[by] * wz[bz]) + (by ? q[1] : -q[1]) * (wx[bx] * wz[bz]) +
                                       (bz ? q[2] : -q[2]) * (wx[bx] * wy[by]));
          const float2 vf = __half22float2(v[u][c8]);
          t0 = fmaf(vf.x, sdot, t0); t1 = fmaf(vf.y, sdot, t1);
          cc0[c8] = fmaf(de[u].x, w, gy0 * sdot); cc1[c8] = fmaf(de[u].y, w, gy1 * sdot);
        }
      }
      if (agg) {
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
          const unsigned rid = __shfl_up_sync(0xffffffffu, run_id, off);
          const bool take = lane >= off && rid == run_id;
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8) {
            const float x0 = __shfl_up_sync(0xffffffffu, cc0[c8], off), x1 = __shfl_up_sync(0xffffffffu, cc1[c8], off);
            if (take) { cc0[c8] += x0; cc1[c8] += x1; }
          }
        }
      }
      if (act && tail) {
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8)
          if (cc0[c8] != 0.f || cc1[c8] != 0.f) atomicAdd(gg + off2[u] + idx[u][c8], make_float2(cc0[c8], cc1[c8]));
      }
      t0 = gs_warp_sum(t0); t1 = gs_warp_sum(t1);
      if (lane == 0 && (t0 != 0.f || t1 != 0.f)) { atomicAdd(a.d_w0 + 3 + 2 * l, t0); atomicAdd(a.d_w0 + 3 + 2 * l + 1, t1); }
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = gs_warp_sum(dw_xyz[c]);
    if (lane == 0 && v != 0.f) atomicAdd(a.d_w0 + c, v);
  }
}


// ------------------------------------------------------------------------------------------------------
// neus_mlp_bwd_kernel — the row-wise half of the colour network's backward in ONE pass per 32-sample warp tile:
// recompute H1 = relu(X W1^T), H2 = relu(H1 W2^T) from the input rows the forward kept, then
//   dH2 = (dY W3) . [H2 > 0],  dH1 = (dH2 W2) . [H1 > 0],  dX = dH1 W1
// on mma.sync (fp16 operands scaled by the loss scale, fp32 accumulation), and everything that hangs off dX per sample:
// the embedding gradient dE = dX[:33] cos(p B), dL/d normal (+ the alpha / eikonal part), dL/d(sdf_layer output), the
// sdf_layer input row h = [x | enc | 1] and the fp16 hi/lo split of the positions.  What is left for cuBLAS are the five
// weight-gradient GEMMs over the sample dimension (A^T B with K = n) and dL/d enc = d_out W_sdf.
// ------------------------------------------------------------------------------------------------------
constexpr int kMbWarps = 8;
constexpr int kW3TPad = 24;          // W3^T row: 16 outputs + padding (48 B rows keep ldmatrix conflict-free)
struct MlpBwdSlab {
  alignas(16) __half a[32 * kInPad];       // X -> dH2 -> dX
  alignas(16) __half b[32 * kHidPad];      // H1
  alignas(16) __half c[32 * kHidPad];      // H2 -> dH1
  alignas(16) __half dy[32 * kW3TPad];     // dY (16 columns, 3 used)
};
struct MlpBwdSmem {
  alignas(16) __half W1[kHid * kInPad];        // [64][80]
  alignas(16) __half W2[kHid * kHidPad];       // [64][64]
  alignas(16) __half W3T[kHid * kW3TPad];      // [64][16]  = W3^T
  alignas(16) __half W2T[kHid * kHidPad];      // [64][64]  = W2^T
  alignas(16) __half W1T[kIn * kHidPad];       // [80][64]  = W1^T
  float colB[3 * 33];
  MlpBwdSlab slab[kMbWarps];
};
struct MlpBwdArgs {
  const __half* mlp_w; const float* color_B;
  const __half* X;                 // [n,80]
  const __half* enc;               // [n,32]
  const float* pos;                // [n,3] normalised position
  const float* d_y;                // [n,3]
  const float* d_s;                // [n]
  const float* d_g;                // [n,3]
  const float* rays_o; const float* rays_d; const float* z_mid;
  const float* scale;              // device scalar (power of two)
  __half* H1; __half* H2; __half* dH1; __half* dH2;    // [n,64]
  __half* dY8;                     // [n,8]
  __half* dE;                      // [n,40]
  __half* d_out;                   // [n,32]
  __half* h;                       // [n,40]: x(3) | enc(32) | 1 | 0...
  __half* pts_hl;                  // [n,8]: hi(3) | lo(3) | 0 0
  float* d_gt;                     // [n,3]
  long long n; int S;
};

template <int NT, int LD>
__device__ __forceinline__ void store_masked_half(const float (&acc)[2][NT][4], const __half* act, __half* out, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int col = nt * 8 + 2 * t;
      const float2 m0 = __half22float2(*reinterpret_cast<const __half2*>(act + (mt * 16 + g) * LD + col));
      const float2 m1 = __half22float2(*reinterpret_cast<const __half2*>(act + (mt * 16 + g + 8) * LD + col));
      const __half2 lo = __floats2half2_rn(m0.x > 0.f ? acc[mt][nt][0] : 0.f, m0.y > 0.f ? acc[mt][nt][1] : 0.f);
      const __half2 hi = __floats2half2_rn(m1.x > 0.f ? acc[mt][nt][2] : 0.f, m1.y > 0.f ? acc[mt][nt][3] : 0.f);
      *reinterpret_cast<__half2*>(out + (mt * 16 + g) * LD + col) = lo;
      *reinterpret_cast<__half2*>(out + (mt * 16 + g + 8) * LD + col) = hi;
    }
}

template <int NT, int LD>
__device__ __forceinline__ void store_half(const float (&acc)[2][NT][4], __half* out, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int col = nt * 8 + 2 * t;
      *reinterpret_cast<__half2*>(out + (mt * 16 + g) * LD + col) = __floats2half2_rn(acc[mt][nt][0], acc[mt][nt][1]);
      *reinterpret_cast<__half2*>(out + (mt * 16 + g + 8) * LD + col) = __floats2half2_rn(acc[mt][nt][2], acc[mt][nt][3]);
    }
}

// copy `bytes` (a multiple of 16) of this lane's row between shared and global memory
__device__ __forceinline__ void copy_row16(void* dst, const void* src, int bytes) {
  uint4* d = reinterpret_cast<uint4*>(dst);
  const uint4* s = reinterpret_cast<const uint4*>(src);
  for (int v = 0; v < bytes / 16; ++v) d[v] = s[v];
}

__global__ void __launch_bounds__(kMbWarps * 32, 1) neus_mlp_bwd_kernel(const MlpBwdArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  MlpBwdSmem& sm = *reinterpret_cast<MlpBwdSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  {
    const __half* w = a.mlp_w;
    for (int i = tid; i < kHid * kIn; i += kMbWarps * 32) {
      const int o = i / kIn, k = i % kIn;
      sm.W1[o * kInPad + k] = w[i];
      sm.W1T[k * kHidPad + o] = w[i];
    }
    for (int i = tid; i < kHid * kHid; i += kMbWarps * 32) {
      const int o = i / kHid, k = i % kHid;
      sm.W2[o * kHidPad + k] = w[kHid * kIn + i];
      sm.W2T[k * kHidPad + o] = w[kHid * kIn + i];
    }
    for (int i = tid; i < kOutW * kHid; i += kMbWarps * 32) {
      const int o = i / kHid, k = i % kHid;
      sm.W3T[k * kW3TPad + o] = w[kHid * kIn + kHid * kHid + i];
    }
    for (int i = tid; i < kHid * (kW3TPad - kOutW); i += kMbWarps * 32)
      sm.W3T[(i / (kW3TPad - kOutW)) * kW3TPad + kOutW + i % (kW3TPad - kOutW)] = __float2half_rn(0.f);
    for (int i = tid; i < 99; i += kMbWarps * 32) sm.colB[i] = a.color_B[i];
  }
  __syncthreads();
  MlpBwdSlab& sl = sm.slab[warp];
  const float sc = __ldg(a.scale), inv_sc = 1.0f / sc;
  const long long ntiles = (a.n + 31) / 32;
  for (long long tile = (long long)blockIdx.x * kMbWarps + warp; tile < ntiles; tile += (long long)gridDim.x * kMbWarps) {
    const long long i = tile * 32 + lane;
    const bool valid = i < a.n;
    // ---- stage X and dY ----
    __half* xrow = sl.a + lane * kInPad;
    if (valid) {
      copy_row16(xrow, a.X + i * kIn, kIn * 2);
    } else {
      for (int k = 0; k < kIn; k += 8) *reinterpret_cast<uint4*>(xrow + k) = make_uint4(0, 0, 0, 0);
    }
    {
      __half* dyr = sl.dy + lane * kW3TPad;
      float y0 = 0.f, y1 = 0.f, y2 = 0.f;
      if (valid) { y0 = a.d_y[i * 3] * sc; y1 = a.d_y[i * 3 + 1] * sc; y2 = a.d_y[i * 3 + 2] * sc; }
      *reinterpret_cast<__half2*>(dyr) = __floats2half2_rn(y0, y1);
      *reinterpret_cast<__half2*>(dyr + 2) = __floats2half2_rn(y2, 0.f);
#pragma unroll
      for (int k = 4; k < kW3TPad; k += 2) *reinterpret_cast<__half2*>(dyr + k) = __float2half2_rn(0.f);
      if (valid) *reinterpret_cast<uint4*>(a.dY8 + i * 8) = *reinterpret_cast<const uint4*>(dyr);
    }
    __syncwarp();
    // ---- forward recompute ----
    {
      float acc[2][8][4];
      warp_layer<8, kIn / 16, kInPad, kInPad>(sl.a, sm.W1, acc, lane);
      store_relu_half<8, kHidPad>(acc, sl.b, lane);
      __syncwarp();
      warp_layer<8, kHid / 16, kHidPad, kHidPad>(sl.b, sm.W2, acc, lane);
      store_relu_half<8, kHidPad>(acc, sl.c, lane);
      __syncwarp();
      if (valid) { copy_row16(a.H1 + i * kHid, sl.b + lane * kHidPad, kHid * 2); copy_row16(a.H2 + i * kHid, sl.c + lane * kHidPad, kHid * 2); }
      // ---- dH2 = (dY W3) . [H2 > 0]  -> sl.a (X is not needed any more) ----
      warp_layer<8, 1, kW3TPad, kW3TPad>(sl.dy, sm.W3T, acc, lane);
      __syncwarp();
      store_masked_half<8, kHidPad>(acc, sl.c, sl.a, lane);       // rows of sl.a re-strided to kHidPad
      __syncwarp();
      if (valid) copy_row16(a.dH2 + i * kHid, sl.a + lane * kHidPad, kHid * 2);
      // ---- dH1 = (dH2 W2) . [H1 > 0]  -> sl.c ----
      warp_layer<8, kHid / 16, kHidPad, kHidPad>(sl.a, sm.W2T, acc, lane);
      __syncwarp();
      store_masked_half<8, kHidPad>(acc, sl.b, sl.c, lane);
      __syncwarp();
      if (valid) copy_row16(a.dH1 + i * kHid, sl.c + lane * kHidPad, kHid * 2);
    }
    // ---- dX = dH1 W1 -> sl.a (stride kInPad) ----
    {
      float accx[2][kIn / 8][4];
      warp_layer<kIn / 8, kHid / 16, kHidPad, kHidPad>(sl.c, sm.W1T, accx, lane);
      __syncwarp();
      store_half<kIn / 8, kInPad>(accx, sl.a, lane);
    }
    __syncwarp();
    // ---- per sample: everything that hangs off this row of dX ----
    if (valid) {
      const __half* dx = sl.a + lane * kInPad;
      const long long ray = i / a.S;
      const float zm = a.z_mid[i];
      float pt[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) pt[c] = __fadd_rn(a.rays_o[ray * 3 + c], __fmul_rn(a.rays_d[ray * 3 + c], zm));
      // embedding: d/d(arg) sin(arg) = cos(arg) = sin(arg + pi/2)
      alignas(16) __half e[40];
#pragma unroll
      for (int j = 0; j < 33; ++j) {
        const float arg = pt[0] * sm.colB[j] + pt[1] * sm.colB[33 + j] + pt[2] * sm.colB[66 + j];
        e[j] = __float2half_rn(__half2float(dx[j]) * fast_sin(arg + 1.57079632679489662f));
      }
#pragma unroll
      for (int j = 33; j < 40; ++j) e[j] = __float2half_rn(0.f);
      copy_row16(a.dE + i * 40, e, 80);
      // normal
#pragma unroll
      for (int c = 0; c < 3; ++c) a.d_gt[i * 3 + c] = a.d_g[i * 3 + c] + __half2float(dx[33 + c]) * inv_sc;
      // sdf_layer output gradient [d sdf | d feat(31)]
      alignas(16) __half o[32];
      o[0] = __float2half_rn(a.d_s[i] * sc);
#pragma unroll
      for (int j = 1; j < 32; ++j) o[j] = dx[35 + j];
      copy_row16(a.d_out + i * 32, o, 64);
      // sdf_layer input row [x | enc | 1 | 0 0 0 0]  (the 1 makes the bias gradient a column of the same GEMM)
      alignas(16) __half hrow[40];
#pragma unroll
      for (int c = 0; c < 3; ++c) hrow[c] = __float2half_rn(a.pos[i * 3 + c]);
      {
        const uint4* es = reinterpret_cast<const uint4*>(a.enc + i * 32);
        uint4 ev[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) ev[v] = es[v];
        const __half* eh = reinterpret_cast<const __half*>(ev);
#pragma unroll
        for (int j = 0; j < 32; ++j) hrow[3 + j] = eh[j];
      }
      hrow[35] = __float2half_rn(1.f);
#pragma unroll
      for (int j = 36; j < 40; ++j) hrow[j] = __float2half_rn(0.f);
      copy_row16(a.h + i * 40, hrow, 80);
      // positions as fp16 hi + lo (exact to 2^-22): the embedding matrix gradient is a GEMM over them
      alignas(16) __half pl[8];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        pl[c] = __float2half_rn(pt[c]);
        pl[3 + c] = __float2half_rn(pt[c] - __half2float(pl[c]));
      }
      pl[6] = pl[7] = __float2half_rn(0.f);
      copy_row16(a.pts_hl + i * 8, pl, 16);
    }
    __syncwarp();
  }
}

// hash-grid constants are per DEVICE (constant memory) and the opt-in shared memory is per device too
cudaError_t neus_device_setup(int) {
  GridMeta g = make_grid_meta(nullptr);
  LevelConst lc[kLevels];
  for (int l = 0; l < kLevels; ++l) {
    lc[l].scale = g.scale[l];
    lc[l].res = (unsigned)g.res[l];
    lc[l].res2 = (unsigned)g.res[l] * (unsigned)g.res[l];
    lc[l].offset = g.offset[l];
    lc[l].size = g.size[l];
    const unsigned long long dense = (unsigned long long)g.res[l] * g.res[l] * g.res[l];
    const bool hashed = dense > g.size[l];
    if (hashed != (l >= kDenseLevels) || (hashed && g.size[l] != (1u << 19))) return cudaErrorInvalidValue;
  }
  cudaError_t e = cudaMemcpyToSymbol(c_lvl, lc, sizeof(lc));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(neus_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(neus_mlp_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(MlpBwdSmem));
  return e;
}

GsDeviceOnce g_neus_once;
int neus_device_init() { return gs_device_once(g_neus_once, neus_device_setup); }

}  // namespace

extern "C" {

int64_t goslam_hashgrid_layout(int64_t* offsets, int* resolutions, float* scales) {
  int64_t total = 0;
  GridMeta g = make_grid_meta(&total);
  for (int l = 0; l < kLevels; ++l) {
    if (offsets) offsets[l] = (int64_t)g.offset[l] * 2;
    if (resolutions) resolutions[l] = g.res[l];
    if (scales) scales[l] = g.scale[l];
  }
  if (offsets) offsets[kLevels] = total * 2;
  return total * 2;
}

size_t goslam_neus_workspace_bytes(int R, int S) {
  (void)R; (void)S;
  return gs_align(148 * 4 * sizeof(float)) + gs_align(148 * 4 * sizeof(unsigned)) + 256;
}

int goslam_neus_forward(const goslam_neus_params* params, const float* rays_o, const float* rays_d,
                        const float* z_vals, const float* dists, int R, int S,
                        const goslam_neus_out* out, void* workspace, size_t workspace_bytes,
                        void* stream) {
  if (!params || !out || R < 0 || S <= 0 || S > kMaxGroup) return GOSLAM_EINVAL;
  if (R == 0) return GOSLAM_OK;
  if (workspace == nullptr || workspace_bytes < goslam_neus_workspace_bytes(R, S))
    return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  { const int rc = neus_device_init(); if (rc != GOSLAM_OK) return rc; }
  GsArena ar(workspace, workspace_bytes);
  NeusArgs a{};
  a.p = *params; a.o = *out;
  a.rays_o = rays_o; a.rays_d = rays_d; a.z_vals = z_vals; a.dists = dists;
  a.R = R; a.S = S;
  const int grid = 148;
  a.blk_gerr = ar.take<float>(148 * 4);
  a.blk_count = ar.take<unsigned>(148 * 4);
  a.flag = reinterpret_cast<int*>(ar.take<int>(1));
  // rays per warp work item: make G*S a multiple of 32 when that fits the slab, else pad
  int G = 32 / std::__gcd(S, 32);
  if (G * S > kMaxGroup) G = kMaxGroup / S;
  if (G < 1) return GOSLAM_EINVAL;
  a.rays_per_group = G;
  const int groups = gs_cdiv(R, G);
  const int nblk = gs_cdiv(groups, kWarpsN) < grid ? gs_cdiv(groups, kWarpsN) : grid;
  for (int mode = 0; mode < 2; ++mode) {
    a.mode = mode;
    neus_forward_kernel<<<nblk, kThreadsN, sizeof(Smem), st>>>(a);
    GS_CHECK_LAUNCH();
    neus_finalize_kernel<<<1, 32, 0, st>>>(a.blk_gerr, a.blk_count, nblk, (long long)R * S,
                                           out->gradient_error, a.flag, mode);
    GS_CHECK_LAUNCH();
  }
  return GOSLAM_OK;
}

int goslam_neus_composite_backward(const goslam_neus_params* params, const float* rays_o, const float* rays_d,
                                   const float* dists, const float* alpha, const float* rgb, const float* sdf,
                                   const float* grad, const float* z_mid, const float* d_color, const float* d_depth,
                                   const float* d_sdf, const float* d_gradient_error, long long total_samples, int R, int S,
                                   float* d_mlp_out, float* d_sdf_out, float* d_grad, float* d_inv_s, void* stream) {
  if (!params || !rays_o || !rays_d || !dists || !alpha || !rgb || !sdf || !grad || !z_mid || !d_mlp_out || !d_sdf_out ||
      !d_grad || !d_inv_s || R < 0 || S <= 0 || S > 32 * kCompChunks || total_samples < (long long)R * S)
    return GOSLAM_EINVAL;
  if (R == 0) return GOSLAM_OK;
  CompBwdArgs a{};
  a.p = *params; a.rays_o = rays_o; a.rays_d = rays_d; a.dists = dists;
  a.alpha = alpha; a.rgb = rgb; a.sdf = sdf; a.grad = grad; a.z_mid = z_mid;
  a.d_color = d_color; a.d_depth = d_depth; a.d_sdf = d_sdf; a.d_gerr = d_gradient_error;
  a.gerr_norm = total_samples > 0 ? (float)(1.0 / (double)total_samples) : 0.f;
  a.d_mlp_out = d_mlp_out; a.d_sdf_out = d_sdf_out; a.d_grad = d_grad; a.d_inv_s = d_inv_s;
  a.R = R; a.S = S;
  neus_composite_bwd_kernel<<<gs_cdiv(R, 8), 256, 0, (cudaStream_t)stream>>>(a);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_neus_mlp_backward(const goslam_neus_params* params, const void* mlp_in, const void* enc, const float* pos,
                             const float* d_mlp_out, const float* d_sdf, const float* d_grad, const float* rays_o,
                             const float* rays_d, const float* z_mid, const float* scale, int R, int S,
                             const goslam_neus_mlp_bwd_out* out, void* stream) {
  if (!params || !mlp_in || !enc || !pos || !d_mlp_out || !d_sdf || !d_grad || !rays_o || !rays_d || !z_mid || !scale || !out ||
      !out->H1 || !out->H2 || !out->dH1 || !out->dH2 || !out->dY8 || !out->dE || !out->d_out || !out->h || !out->pts_hl ||
      !out->d_grad_total || R < 0 || S <= 0)
    return GOSLAM_EINVAL;
  if (R == 0) return GOSLAM_OK;
  { const int rc = neus_device_init(); if (rc != GOSLAM_OK) return rc; }
  MlpBwdArgs a{};
  a.mlp_w = reinterpret_cast<const __half*>(params->mlp_w); a.color_B = params->color_B;
  a.X = reinterpret_cast<const __half*>(mlp_in); a.enc = reinterpret_cast<const __half*>(enc); a.pos = pos;
  a.d_y = d_mlp_out; a.d_s = d_sdf; a.d_g = d_grad; a.rays_o = rays_o; a.rays_d = rays_d; a.z_mid = z_mid; a.scale = scale;
  a.H1 = reinterpret_cast<__half*>(out->H1); a.H2 = reinterpret_cast<__half*>(out->H2);
  a.dH1 = reinterpret_cast<__half*>(out->dH1); a.dH2 = reinterpret_cast<__half*>(out->dH2);
  a.dY8 = reinterpret_cast<__half*>(out->dY8); a.dE = reinterpret_cast<__half*>(out->dE);
  a.d_out = reinterpret_cast<__half*>(out->d_out); a.h = reinterpret_cast<__half*>(out->h);
  a.pts_hl = reinterpret_cast<__half*>(out->pts_hl); a.d_gt = out->d_grad_total;
  a.n = (long long)R * S; a.S = S;
  const long long tiles = (a.n + 31) / 32;
  const long long blocks = (tiles + kMbWarps - 1) / kMbWarps;
  neus_mlp_bwd_kernel<<<(unsigned)(blocks < 148 ? blocks : 148), kMbWarps * 32, sizeof(MlpBwdSmem), (cudaStream_t)stream>>>(a);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_neus_grid_backward(const goslam_neus_params* params, const float* rays_o, const float* rays_d,
                              const float* z_vals, const float* dists, int R, int S, const float* d_enc,
                              const float* d_enc_scale, const float* d_grad, float* grid_grad, float* d_w0, void* stream) {
  if (!params || !rays_o || !rays_d || !z_vals || !dists || !d_enc || !d_grad || !grid_grad || !d_w0 || R < 0 || S <= 0)
    return GOSLAM_EINVAL;
  if (R == 0) return GOSLAM_OK;
  { const int rc = neus_device_init(); if (rc != GOSLAM_OK) return rc; }
  GridBwdArgs a{};
  a.p = *params; a.rays_o = rays_o; a.rays_d = rays_d; a.z_vals = z_vals; a.dists = dists;
  a.d_enc = d_enc; a.d_enc_scale = d_enc_scale; a.d_grad = d_grad; a.grid_grad = grid_grad; a.d_w0 = d_w0;
  a.n = (long long)R * S; a.S = S;
  const long long blocks = (a.n + 255) / 256;
  if (blocks > 0x7fffffffLL) return GOSLAM_EINVAL;
  neus_grid_bwd_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

}  // extern "C"
