// corr_build_tc.cu — all-pairs correlation volume on Blackwell tensor cores (tcgen05 + TMA)
// with the 4-level average-pool pyramid produced in the epilogue.
//
// Reference: CorrBlock.__init__ / CorrBlock.corr (src/modules/corr.py:25-41,67-76) —
// torch.matmul (cuBLAS) writes level 0, then three F.avg_pool2d passes re-read the volume.
//
// Design (one CTA per SM, persistent, warp-specialised, 576 threads):
//   warp 0      TMA producer: A tile = 128 source pixels x 128 channels (2 boxes of 64 ch,
//               128B-swizzled, K-major) once per work item (edge, source tile, 8-row target band);
//               B tile = an 8x16 patch of TARGET pixels x 128 channels (4-D tensor map
//               (ch, x, y, slot) -> rows ordered y*16+x), 2-stage ring.  Out-of-image rows/cols are
//               zero-filled by TMA.  Feature maps are indexed per edge on the device
//               (slot1 = rig*ii, slot2 = rig*jj + (ii==jj)), so no gathered copies exist.
//   warp 1      MMA issuer: 8 x tcgen05.mma (M128,N128,K16, fp16 in / fp32 accumulate in TMEM) per
//               tile, 2 accumulator stages (256 TMEM columns); tcgen05.commit -> mbarriers.
//   warps 2-17  epilogue, two groups of 8 (one per TMEM stage).  Two warps share a TMEM lane
//               quadrant and split the tile's columns (= patch rows 0-3 / 4-7), so 16 warps keep
//               TMEM reads, conversions and global stores of two tiles in flight.  A thread owns
//               4 rows x 16 columns of its source pixel's patch: fp16 rounding, level 0 as
//               full-sector 256-bit stores, levels 1-2 pooled in registers FROM THE ROUNDED finer
//               level (the avg_pool2d numerics) and staged in shared memory per band; when the
//               band's x-tiles are done the pooled rows (and level 3, pooled from the staged
//               level 2) leave as long contiguous runs.  The volume is never re-read.
// Why the band staging: partial 32-byte-sector writes cost an ECC read-modify-write in L2 and
// were measured to cost more than all of level 0 (profiles/r01_corr_build_notes.md).
// The 1/4 feature scaling of the reference (`fmap / 4.0` in half) is applied by the K-major
// re-layout prepass, exactly as the reference does it, so the accumulator needs no scaling.
#include "common.cuh"
#include "launch.cuh"
#include "tc_ptx.cuh"
#include <cstdio>

int gs_corr_build_simt_f16(const __half* f1, const __half* f2, __half* const* levels,
                           int num_levels, int N, int D, int h, int w, cudaStream_t st);

namespace {

constexpr int kD = 128;                 // channels (K)
constexpr int kBM = 128;                // source pixels per tile
constexpr int kPY = 8, kPX = 16;        // target patch
constexpr int kBN = kPY * kPX;          // 128
constexpr int kKBox = 64;               // channels per TMA box (128 B)
constexpr int kTileBytes = kBM * kD * 2;          // 32 KB (A or B tile)
constexpr int kBoxBytes = kBM * kKBox * 2;        // 16 KB
constexpr int kAStages = 2, kBStages = 2, kTStages = 2;
constexpr int kEpiWarps = 8;                      // per group (2 per TMEM lane quadrant)
constexpr int kEpiThreads = kTStages * kEpiWarps * 32;   // 512
constexpr int kThreadsTC = 64 + kEpiThreads;             // 576
constexpr int kMaxXB = 8;                                // x-tiles per band (w <= 128)
constexpr int kPoolMax = kBM * ((4 * kMaxXB * 16 + 16) + (2 * kMaxXB * 8 + 8));   // 84,992 B (level 1 | level 2 pieces)
constexpr int kSmemTC = 1024 + (kAStages + kBStages) * kTileBytes + kPoolMax + 256;

using namespace gs_tc;

// kind::f16 instruction descriptor: D=f32 (bits 4-5 = 1), A=B=f16 (0), both K-major,
// N>>3 at bits 17-22, M>>4 at bits 24-28.
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);

struct TcParams {
  __half* lvl[4];
  int num_levels, N, h, w, hw;
  int n_mt, n_yb, n_xb;       // m-tiles, y-blocks, x-blocks
  int n_items;                // N * n_mt * n_yb
  // optional edge -> feature-map-slot indirection (video-level K-major feature maps):
  // slot1 = rig*ii[e], slot2 = rig*jj[e] + (ii[e]==jj[e])   (src/factor_graph.py:108-113,290)
  const int64_t* ii; const int64_t* jj; int rig;
  const int* out_slot;        // optional edge -> output slot of the level buffers (CorrPool)
  // tiled = 1: levels 0 and 1 are stored as 4x4-element (32-byte) tiles, tile-row-major inside each
  // source pixel's plane (plane = H4*W4 tiles, padded with zeros); levels 2, 3 stay row-major.
  int tiled, w4_0, h4_0, w4_1, h4_1;
  int pitch2, pitch3;         // tiled: bytes per (source pixel, band) of levels 2 / 3 (multiples of 32)
  int aligned;                // w % 16 == 0 && h % 8 == 0: every store is a whole aligned sector run
};

// ---- packed fp16 rows live in registers as uint32 pairs (lo = even column) ----
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}
__device__ __forceinline__ float lo_f(uint32_t u) {
  return __half2float(__ushort_as_half((unsigned short)(u & 0xffffu)));
}
__device__ __forceinline__ float hi_f(uint32_t u) {
  return __half2float(__ushort_as_half((unsigned short)(u >> 16)));
}
// 2x2 mean of ROUNDED halves, fp32 sum in row-major window order, one rounding (avg_pool2d)
__device__ __forceinline__ float pool_pair(uint32_t top, uint32_t bot) {
  float s = lo_f(top);
  s += hi_f(top);
  s += lo_f(bot);
  s += hi_f(bot);
  return s * 0.25f;
}
// store NW packed words (2*NW halves) to dst, honouring alignment and the valid count
template <int NW>
__device__ __forceinline__ void store_row(__half* dst, const uint32_t (&r)[NW], int nvalid) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(dst);
  if (nvalid >= 2 * NW) {
    if (NW == 8 && (a & 31) == 0) {     // one full 32-byte sector per lane (STG.256)
      asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "r"(r[0]),
                   "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                   : "memory");
      return;
    }
    if (NW >= 4 && (a & 15) == 0) {
#pragma unroll
      for (int i = 0; i < NW; i += 4)
        *reinterpret_cast<uint4*>(dst + 2 * i) = make_uint4(r[i], r[i + 1], r[i + 2], r[i + 3]);
      return;
    }
    if (NW == 2 && (a & 7) == 0) {
      *reinterpret_cast<uint2*>(dst) = make_uint2(r[0], r[1]);
      return;
    }
    if ((a & 3) == 0) {
#pragma unroll
      for (int i = 0; i < NW; ++i) *reinterpret_cast<uint32_t*>(dst + 2 * i) = r[i];
      return;
    }
  }
#pragma unroll
  for (int i = 0; i < NW; ++i) {
    if (2 * i < nvalid) dst[2 * i] = __ushort_as_half((unsigned short)(r[i] & 0xffffu));
    if (2 * i + 1 < nvalid) dst[2 * i + 1] = __ushort_as_half((unsigned short)(r[i] >> 16));
  }
}

__global__ void __launch_bounds__(kThreadsTC, 1)
corr_build_tc_kernel(const __grid_constant__ CUtensorMap mapA,
                     const __grid_constant__ CUtensorMap mapB, const TcParams p) {
  extern __shared__ unsigned char smem_raw[];
  // 1024-byte alignment for the 128B swizzle atoms
  unsigned char* base =
      reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smA = base;
  unsigned char* smB = base + kAStages * kTileBytes;
  unsigned char* smPool = base + (kAStages + kBStages) * kTileBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smPool + kPoolMax);
  uint64_t* full_a = bars;                       // [kAStages]
  uint64_t* empty_a = full_a + kAStages;
  uint64_t* full_b = empty_a + kAStages;         // [kBStages]
  uint64_t* empty_b = full_b + kBStages;
  uint64_t* tm_full = empty_b + kBStages;        // [kTStages]
  uint64_t* tm_empty = tm_full + kTStages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tm_empty + kTStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kAStages; ++i) { mbar_init(&full_a[i], 1); mbar_init(&empty_a[i], 1); }
    for (int i = 0; i < kBStages; ++i) { mbar_init(&full_b[i], 1); mbar_init(&empty_b[i], 1); }
    for (int i = 0; i < kTStages; ++i) { mbar_init(&tm_full[i], 1); mbar_init(&tm_empty[i], kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, kTStages * kBN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int as = 0, aph = 0, bs = 0, bph = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int yb = item % p.n_yb;
        const int mt = (item / p.n_yb) % p.n_mt;
        const int n = item / (p.n_yb * p.n_mt);
        int n1 = n, n2 = n;
        if (p.ii != nullptr) {
          const int fi = (int)p.ii[n], fj = (int)p.jj[n];
          n1 = p.rig * fi;
          n2 = p.rig * fj + ((fi == fj && p.rig > 1) ? 1 : 0);
        }
        mbar_wait(&empty_a[as], aph ^ 1);
        mbar_expect_tx(&full_a[as], kTileBytes);
        tma_load_3d(&mapA, &full_a[as], smA + as * kTileBytes, 0, mt * kBM, n1);
        tma_load_3d(&mapA, &full_a[as], smA + as * kTileBytes + kBoxBytes, kKBox, mt * kBM, n1);
        if (++as == kAStages) { as = 0; aph ^= 1; }
        for (int xb = 0; xb < p.n_xb; ++xb) {
          mbar_wait(&empty_b[bs], bph ^ 1);
          mbar_expect_tx(&full_b[bs], kTileBytes);
          tma_load_4d(&mapB, &full_b[bs], smB + bs * kTileBytes, 0, xb * kPX, yb * kPY, n2);
          tma_load_4d(&mapB, &full_b[bs], smB + bs * kTileBytes + kBoxBytes, kKBox, xb * kPX,
                      yb * kPY, n2);
          if (++bs == kBStages) { bs = 0; bph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int as = 0, aph = 0, bs = 0, bph = 0, ts = 0, tph = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        mbar_wait(&full_a[as], aph);
        const uint32_t a_addr = smem_u32(smA + as * kTileBytes);
        for (int xb = 0; xb < p.n_xb; ++xb) {
          mbar_wait(&tm_empty[ts], tph ^ 1);
          mbar_wait(&full_b[bs], bph);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(smB + bs * kTileBytes);
          const uint32_t d_tmem = tmem_base + ts * kBN;
#pragma unroll
          for (int kb = 0; kb < kD / kKBox; ++kb) {
#pragma unroll
            for (int k = 0; k < kKBox / 16; ++k) {
              const uint64_t da = make_desc_sw128(a_addr + kb * kBoxBytes + k * 32);
              const uint64_t db = make_desc_sw128(b_addr + kb * kBoxBytes + k * 32);
              umma_f16(d_tmem, da, db, kIdesc, (kb | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(&empty_b[bs]);      // smem B stage reusable when these MMAs retire
          umma_commit(&tm_full[ts]);      // accumulator ready for the epilogue
          if (++bs == kBStages) { bs = 0; bph ^= 1; }
          if (++ts == kTStages) { ts = 0; tph ^= 1; }
        }
        umma_commit(&empty_a[as]);
        if (++as == kAStages) { as = 0; aph ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (warps 2..17) =====================
    const int ew = warp - 2;                      // 0..15
    const int group = ew >> 3;                    // TMEM stage this warp drains
    const int wq = ew & 7;
    const int quad = warp & 3;                    // TMEM lane quadrant a warp may read = warp_id % 4
    const int half = wq >> 2;                     // patch rows 4*half .. 4*half+3 (columns 64*half..)
    const int row = quad * 32 + lane;             // row of the 128-row tile = source pixel
    const int etid = threadIdx.x - 64;            // 0..511
    const int ts = group;
    // band staging strides (bytes); the +16 / +8 pads make the per-source-pixel stride conflict-free
    const int p1row = p.n_xb * 16, p1src = 4 * p1row + 16;
    const int p2row = p.n_xb * 8;
    const int p2src = p.tiled ? p.pitch2 + 8 : 2 * p2row + 8;
    unsigned char* pool1 = smPool;
    unsigned char* pool2 = smPool + kBM * p1src;
    const int h1 = p.h >> 1, w1 = p.w >> 1, h2 = p.h >> 2, w2 = p.w >> 2, h3 = p.h >> 3, w3 = p.w >> 3;
    int tph = 0, tile = 0;
#ifdef GOSLAM_TC_PROBE
    long long pr_wait = 0, pr_tiles = 0, pr_bar1 = 0, pr_wo = 0, pr_bar2 = 0, pr_t0 = clock64();
    const bool pr_on = (etid == 0 || etid == 256) && blockIdx.x == 0;
#define TCP(x) x
#else
#define TCP(x)
#endif
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      TCP(const long long ta = clock64();)
      const int yb = item % p.n_yb;
      const int mt = (item / p.n_yb) % p.n_mt;
      const int n = item / (p.n_yb * p.n_mt);
      const int src = mt * kBM + row;
      const bool src_ok = src < p.hw;
      const int n_out = p.out_slot ? __ldg(p.out_slot + n) : n;
      const long long plane_id = (long long)n_out * p.hw + src;
      const int y0 = yb * kPY;
      for (int xb = 0; xb < p.n_xb; ++xb, ++tile) {
        if ((tile & (kTStages - 1)) != ts) continue;
        const int x0 = xb * kPX;
        TCP(const long long tw = clock64();)
        mbar_wait(&tm_full[ts], tph);
        TCP(pr_wait += clock64() - tw;)
        tc_fence_after();
        const uint32_t taddr = tmem_base + ts * kBN + ((uint32_t)(quad * 32) << 16);
        uint32_t l1[2][4];     // the two level-1 rows this thread produces (8 halves each)
        if (p.tiled) {
          // ---- tiled layout: this thread's 4 patch rows x 16 columns are exactly four 4x4 tiles,
          // adjacent in memory: one 128-byte run per thread (4 x STG.256) ----
          uint32_t hr[4][8];
          {
            uint32_t va[32], vb[32];
            tmem_ld32_issue(taddr + (2 * half) * 32, va);
            tmem_ld32_issue(taddr + (2 * half + 1) * 32, vb);
            tmem_ld_wait();
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
              for (int x = 0; x < 8; ++x) {
                hr[r][x] = pack2(__uint_as_float(va[r * 16 + 2 * x]), __uint_as_float(va[r * 16 + 2 * x + 1]));
                hr[2 + r][x] = pack2(__uint_as_float(vb[r * 16 + 2 * x]), __uint_as_float(vb[r * 16 + 2 * x + 1]));
              }
          }
          // this warp's part of the accumulator stage is in registers: hand it back before storing
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tm_empty[ts]);
          const int ty = 2 * yb + half;
          if (src_ok && ty < p.h4_0) {
            unsigned char* dst = reinterpret_cast<unsigned char*>(p.lvl[0]) +
                                 ((plane_id * p.h4_0 + ty) * p.w4_0 + xb * 4) * 32LL;
#pragma unroll
            for (int t = 0; t < 4; ++t)
              if (xb * 4 + t < p.w4_0)
                asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst + t * 32),
                             "r"(hr[0][2 * t]), "r"(hr[0][2 * t + 1]), "r"(hr[1][2 * t]), "r"(hr[1][2 * t + 1]),
                             "r"(hr[2][2 * t]), "r"(hr[2][2 * t + 1]), "r"(hr[3][2 * t]), "r"(hr[3][2 * t + 1])
                             : "memory");
          }
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              l1[cc][j] = pack2(pool_pair(hr[2 * cc][2 * j], hr[2 * cc + 1][2 * j]),
                                pool_pair(hr[2 * cc][2 * j + 1], hr[2 * cc + 1][2 * j + 1]));
            // level-1 row (2*half+cc) of the band, columns 8*xb .. 8*xb+7 = sub-row of two 4x4 tiles
            unsigned char* st = pool1 + row * p1src + (2 * half + cc) * 8;
            *reinterpret_cast<uint2*>(st + (xb * 2) * 32) = make_uint2(l1[cc][0], l1[cc][1]);
            *reinterpret_cast<uint2*>(st + (xb * 2 + 1) * 32) = make_uint2(l1[cc][2], l1[cc][3]);
          }
        } else {
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int c = 2 * half + cc;           // 32-column chunk = patch rows 2c, 2c+1
          uint32_t v[32];
          tmem_ld32(taddr + c * 32, v);
          uint32_t h0[2][8];
#pragma unroll
          for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int x = 0; x < 8; ++x)
              h0[r][x] = pack2(__uint_as_float(v[r * 16 + 2 * x]), __uint_as_float(v[r * 16 + 2 * x + 1]));
          if (src_ok) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
              const int y = y0 + 2 * c + r;
              if (y < p.h) store_row<8>(p.lvl[0] + (plane_id * p.h + y) * p.w + x0, h0[r], p.w - x0);
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            l1[cc][j] = pack2(pool_pair(h0[0][2 * j], h0[1][2 * j]),
                              pool_pair(h0[0][2 * j + 1], h0[1][2 * j + 1]));
          *reinterpret_cast<uint4*>(pool1 + row * p1src + c * p1row + xb * 16) =
              make_uint4(l1[cc][0], l1[cc][1], l1[cc][2], l1[cc][3]);
        }
        }
        // all TMEM reads of this warp for this stage are complete (tmem_ld32 waits): hand it back
        if (!p.tiled) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tm_empty[ts]);
        }
        // level-2 row `half` of the band, from the two level-1 rows
        {
          const uint32_t a0 = pack2(pool_pair(l1[0][0], l1[1][0]), pool_pair(l1[0][1], l1[1][1]));
          const uint32_t a1 = pack2(pool_pair(l1[0][2], l1[1][2]), pool_pair(l1[0][3], l1[1][3]));
          *reinterpret_cast<uint2*>(pool2 + row * p2src + half * p2row + xb * 8) = make_uint2(a0, a1);
        }
        tph ^= 1;
      }
      // ---- band write-out: all 16 epilogue warps have staged every x-tile of this 8-row band ----
      TCP(const long long tb = clock64(); pr_tiles += tb - ta;)
      asm volatile("bar.sync 3, 512;" ::: "memory");
      TCP(const long long tc = clock64(); pr_bar1 += tc - tb;)
      if (p.num_levels > 1) {
        const int s_loc = etid >> 2, part = etid & 3;          // four threads per source pixel
        const int s_glb = mt * kBM + s_loc;
        if (s_glb < p.hw) {
          const long long pl = (long long)n_out * p.hw + s_glb;
          const unsigned char* sp1 = pool1 + s_loc * p1src;
          const unsigned char* sp2 = pool2 + s_loc * p2src;
          if (p.tiled) {
            // level 1: one tile-row of 4x4 tiles = w4_1 contiguous sectors, already in tile order
            if (yb < p.h4_1) {
              unsigned char* g1 = reinterpret_cast<unsigned char*>(p.lvl[1]) +
                                  ((pl * p.h4_1 + yb) * p.w4_1) * 32LL;
              for (int off = part * 32; off < p.w4_1 * 32; off += 128) {
                uint32_t rr[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) rr[k] = *reinterpret_cast<const uint32_t*>(sp1 + off + 4 * k);
                asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g1 + off), "r"(rr[0]),
                             "r"(rr[1]), "r"(rr[2]), "r"(rr[3]), "r"(rr[4]), "r"(rr[5]), "r"(rr[6]), "r"(rr[7])
                             : "memory");
              }
            }
            // levels 2 / 3: one padded, sector-aligned piece per (source pixel, band): whole sectors only
            if (part == 1 && p.num_levels > 2 && 2 * yb < h2) {
              unsigned char* g2 = reinterpret_cast<unsigned char*>(p.lvl[2]) + (pl * p.n_yb + yb) * (long long)p.pitch2;
              for (int off = 0; off < p.pitch2; off += 32) {
                uint32_t rr[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) rr[k] = *reinterpret_cast<const uint32_t*>(sp2 + off + 4 * k);
                asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g2 + off), "r"(rr[0]),
                             "r"(rr[1]), "r"(rr[2]), "r"(rr[3]), "r"(rr[4]), "r"(rr[5]), "r"(rr[6]), "r"(rr[7])
                             : "memory");
              }
            }
            if (part == 2 && p.num_levels > 3 && yb < h3) {
              uint32_t rr[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) {                    // level-3 columns 2k, 2k+1 of this band's row
                rr[k] = 0u;
                if (k < p.n_xb) {
                  const uint32_t t = *reinterpret_cast<const uint32_t*>(sp2 + 8 * k);
                  const uint32_t t2 = *reinterpret_cast<const uint32_t*>(sp2 + 8 * k + 4);
                  const uint32_t b = *reinterpret_cast<const uint32_t*>(sp2 + p2row + 8 * k);
                  const uint32_t b2 = *reinterpret_cast<const uint32_t*>(sp2 + p2row + 8 * k + 4);
                  rr[k] = pack2(pool_pair(t, b), pool_pair(t2, b2));
                }
              }
              unsigned char* g3 = reinterpret_cast<unsigned char*>(p.lvl[3]) + (pl * p.n_yb + yb) * 32LL;
              asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g3), "r"(rr[0]),
                           "r"(rr[1]), "r"(rr[2]), "r"(rr[3]), "r"(rr[4]), "r"(rr[5]), "r"(rr[6]), "r"(rr[7])
                           : "memory");
            }
          } else if (p.aligned) {
            // level 1: 4 full rows, contiguous in memory, 32-byte aligned: whole sectors
            unsigned char* g1 = reinterpret_cast<unsigned char*>(p.lvl[1]) +
                                (pl * h1 + (y0 >> 1)) * (long long)p1row;
            for (int off = part * 32; off < 4 * p1row; off += 128) {
              uint32_t rr[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) rr[k] = *reinterpret_cast<const uint32_t*>(sp1 + off + 4 * k);
              asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g1 + off), "r"(rr[0]),
                           "r"(rr[1]), "r"(rr[2]), "r"(rr[3]), "r"(rr[4]), "r"(rr[5]), "r"(rr[6]), "r"(rr[7])
                           : "memory");
            }
            if (part == 1 && p.num_levels > 2) {                // level 2: 2 rows, 16-byte chunks
              unsigned char* g2 = reinterpret_cast<unsigned char*>(p.lvl[2]) +
                                  (pl * h2 + (y0 >> 2)) * (long long)p2row;
              for (int off = 0; off < 2 * p2row; off += 16)
                *reinterpret_cast<uint4*>(g2 + off) = make_uint4(
                    *reinterpret_cast<const uint32_t*>(sp2 + off), *reinterpret_cast<const uint32_t*>(sp2 + off + 4),
                    *reinterpret_cast<const uint32_t*>(sp2 + off + 8), *reinterpret_cast<const uint32_t*>(sp2 + off + 12));
            }
            if (part == 2 && p.num_levels > 3) {                // level 3: 1 row pooled from level 2
              __half* g3 = p.lvl[3] + (pl * h3 + (y0 >> 3)) * w3;
              for (int x = 0; x < w3; x += 2) {
                const uint32_t t = *reinterpret_cast<const uint32_t*>(sp2 + 4 * x);        // row 0: cols 2x, 2x+1
                const uint32_t t2 = *reinterpret_cast<const uint32_t*>(sp2 + 4 * x + 4);   //        cols 2x+2, 2x+3
                const uint32_t b = *reinterpret_cast<const uint32_t*>(sp2 + p2row + 4 * x);
                const uint32_t b2 = *reinterpret_cast<const uint32_t*>(sp2 + p2row + 4 * x + 4);
                *reinterpret_cast<uint32_t*>(g3 + x) = pack2(pool_pair(t, b), pool_pair(t2, b2));
              }
            }
          } else {
            // ragged shapes: element-wise with bounds (staging rows are n_xb*8 / n_xb*4 halves wide)
            const __half* s1 = reinterpret_cast<const __half*>(sp1);
            const __half* s2 = reinterpret_cast<const __half*>(sp2);
            for (int r = 0; r < 4; ++r) {
              const int y = (y0 >> 1) + r;
              if (y >= h1) break;
              __half* g = p.lvl[1] + (pl * h1 + y) * w1;
              for (int x = part; x < w1; x += 4) g[x] = s1[r * (p1row / 2) + x];
            }
            if (p.num_levels > 2)
              for (int r = 0; r < 2; ++r) {
                const int y = (y0 >> 2) + r;
                if (y >= h2) break;
                __half* g = p.lvl[2] + (pl * h2 + y) * w2;
                for (int x = part; x < w2; x += 4) g[x] = s2[r * (p2row / 2) + x];
              }
            if (p.num_levels > 3 && (y0 >> 3) < h3) {
              __half* g = p.lvl[3] + (pl * h3 + (y0 >> 3)) * w3;
              for (int x = part; x < w3; x += 4) {
                float sum = __half2float(s2[2 * x]);
                sum += __half2float(s2[2 * x + 1]);
                sum += __half2float(s2[(p2row / 2) + 2 * x]);
                sum += __half2float(s2[(p2row / 2) + 2 * x + 1]);
                g[x] = __float2half_rn(sum * 0.25f);
              }
            }
          }
        }
      }
      TCP(const long long td = clock64(); pr_wo += td - tc;)
      asm volatile("bar.sync 3, 512;" ::: "memory");
      TCP(pr_bar2 += clock64() - td;)
    }
#ifdef GOSLAM_TC_PROBE
    if (pr_on)
      printf("[tc probe etid=%d] total %lld | tile loop %lld (of which tm_full wait %lld) | bar1 %lld | write-out %lld | bar2 %lld\n",
             etid, clock64() - pr_t0, pr_tiles, pr_wait, pr_bar1, pr_wo, pr_bar2);
#endif
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTStages * kBN);
}

// ------------------------------------------------------------------------------------------------------
// Staged variant (tiled slot-pool layout, w <= 80): the write stream is DECOUPLED from the TMEM drain.
//   warp 0 TMA producer | warp 1 MMA issuer | warps 2..9 drain warps (stage = (warp-2)/4, TMEM lane quadrant = warp%4):
//   tcgen05.ld, fp16 conversion, pyramid pooling; they only write SHARED memory (a level-0 slot per TMEM stage, the band
//   pool for levels 1-3) | warps 10..13 store warps: thread = source pixel, they move the staged level-0 tiles (two
//   128-byte runs per tile) and, at the end of a band, the pooled pieces to global memory as whole 32-byte sectors.
// Why: tools/wbench.cu (profiles/r02_wbench_v2.txt) — this very store pattern streams at 6.19 TB/s from 128 threads per
// SM but at 4.92 TB/s from 512, and the direct-store kernel, whose 512 epilogue threads also sit in the store queue
// instead of draining accumulators, ends at (no-write floor 116 µs) + (pure-store time 150 µs) = 283 µs.
// 448 threads: no register cap below the direct-store kernel's 90.
// ------------------------------------------------------------------------------------------------------
constexpr int kDrainWarps = 8, kStoreWarps = 4;
constexpr int kThreadsST = 64 + (kDrainWarps + kStoreWarps) * 32;      // 448
constexpr int kStageRow = 2 * 128 + 16;                                // staged level-0 bytes per source pixel and tile
constexpr int kStageBytes = kBM * kStageRow;                           // 34,816 B per slot (one slot per TMEM stage)
inline int pool_bytes_st(int n_xb) { return kBM * ((4 * n_xb * 16 + 16) + (((n_xb * 16 + 31) / 32 * 32) + 8)); }
inline int smem_staged(int n_xb) { return 1024 + (1 + kBStages) * kTileBytes + pool_bytes_st(n_xb) + kTStages * kStageBytes + 256; }

__global__ void __launch_bounds__(kThreadsST, 1)
corr_build_tc_staged_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                            const TcParams p, const int pool_bytes) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base =
      reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* smA = base;                                   // ONE A stage (reloaded once per 8-row band item)
  unsigned char* smB = base + kTileBytes;
  unsigned char* smPool = base + (1 + kBStages) * kTileBytes;
  unsigned char* smStage = smPool + pool_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smStage + kTStages * kStageBytes);
  uint64_t* full_a = bars;
  uint64_t* empty_a = bars + 1;
  uint64_t* full_b = bars + 2;          // [kBStages]
  uint64_t* empty_b = full_b + kBStages;
  uint64_t* tm_full = empty_b + kBStages;
  uint64_t* tm_empty = tm_full + kTStages;
  uint64_t* st_full = tm_empty + kTStages;      // slot written by its 4 drain warps
  uint64_t* st_empty = st_full + kTStages;      // slot moved out by the 4 store warps
  uint64_t* band_full = st_empty + kTStages;    // pooled pieces of a band complete (8 drain warps)
  uint64_t* band_empty = band_full + 1;         // pool may be overwritten (4 store warps)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(band_empty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(full_a, 1); mbar_init(empty_a, 1);
    for (int i = 0; i < kBStages; ++i) { mbar_init(&full_b[i], 1); mbar_init(&empty_b[i], 1); }
    for (int i = 0; i < kTStages; ++i) {
      mbar_init(&tm_full[i], 1); mbar_init(&tm_empty[i], 4);
      mbar_init(&st_full[i], 4); mbar_init(&st_empty[i], kStoreWarps);
    }
    mbar_init(band_full, kDrainWarps); mbar_init(band_empty, kStoreWarps);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, kTStages * kBN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  const int p1row = p.n_xb * 16, p1src = 4 * p1row + 16;
  const int p2row = p.n_xb * 8, p2src = p.pitch2 + 8;
  unsigned char* pool1 = smPool;
  unsigned char* pool2 = smPool + kBM * p1src;
  const int h2 = p.h >> 2, h3 = p.h >> 3;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int aph = 0, bs = 0, bph = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int yb = item % p.n_yb;
        const int mt = (item / p.n_yb) % p.n_mt;
        const int n = item / (p.n_yb * p.n_mt);
        int n1 = n, n2 = n;
        if (p.ii != nullptr) {
          const int fi = (int)p.ii[n], fj = (int)p.jj[n];
          n1 = p.rig * fi;
          n2 = p.rig * fj + ((fi == fj && p.rig > 1) ? 1 : 0);
        }
        mbar_wait(empty_a, aph ^ 1);
        mbar_expect_tx(full_a, kTileBytes);
        tma_load_3d(&mapA, full_a, smA, 0, mt * kBM, n1);
        tma_load_3d(&mapA, full_a, smA + kBoxBytes, kKBox, mt * kBM, n1);
        aph ^= 1;
        for (int xb = 0; xb < p.n_xb; ++xb) {
          mbar_wait(&empty_b[bs], bph ^ 1);
          mbar_expect_tx(&full_b[bs], kTileBytes);
          tma_load_4d(&mapB, &full_b[bs], smB + bs * kTileBytes, 0, xb * kPX, yb * kPY, n2);
          tma_load_4d(&mapB, &full_b[bs], smB + bs * kTileBytes + kBoxBytes, kKBox, xb * kPX, yb * kPY, n2);
          if (++bs == kBStages) { bs = 0; bph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int aph = 0, bs = 0, bph = 0, ts = 0, tph = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        mbar_wait(full_a, aph);
        const uint32_t a_addr = smem_u32(smA);
        for (int xb = 0; xb < p.n_xb; ++xb) {
          mbar_wait(&tm_empty[ts], tph ^ 1);
          mbar_wait(&full_b[bs], bph);
          tc_fence_after();
          const uint32_t b_addr = smem_u32(smB + bs * kTileBytes);
          const uint32_t d_tmem = tmem_base + ts * kBN;
#pragma unroll
          for (int kb = 0; kb < kD / kKBox; ++kb)
#pragma unroll
            for (int k = 0; k < kKBox / 16; ++k)
              umma_f16(d_tmem, make_desc_sw128(a_addr + kb * kBoxBytes + k * 32), make_desc_sw128(b_addr + kb * kBoxBytes + k * 32),
                       kIdesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_b[bs]);
          umma_commit(&tm_full[ts]);
          if (++bs == kBStages) { bs = 0; bph ^= 1; }
          if (++ts == kTStages) { ts = 0; tph ^= 1; }
        }
        umma_commit(empty_a);
        aph ^= 1;
      }
    }
  } else if (warp < 2 + kDrainWarps) {
    // ===================== drain warps =====================
    const int ts = (warp - 2) >> 2;               // TMEM stage = staging slot of this warp
    const int quad = warp & 3;                    // TMEM lane quadrant a warp may read = warp_id % 4
    const int row = quad * 32 + lane;             // source pixel of the tile
    unsigned char* slot = smStage + ts * kStageBytes + row * kStageRow;
    int tph = 0, sph = 0, tile = 0, band = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++band) {
      bool pool_ok = false;                       // the store warps have finished the previous band's write-out
      for (int xb = 0; xb < p.n_xb; ++xb, ++tile) {
        if ((tile & (kTStages - 1)) != ts) continue;
        mbar_wait(&tm_full[ts], tph);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ts * kBN + ((uint32_t)(quad * 32) << 16);
        mbar_wait(&st_empty[ts], sph ^ 1);        // slot free (first use passes)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t hr[4][8];
          {
            uint32_t va[32], vb[32];
            tmem_ld32_issue(taddr + (2 * half) * 32, va);
            tmem_ld32_issue(taddr + (2 * half + 1) * 32, vb);
            tmem_ld_wait();
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
              for (int x = 0; x < 8; ++x) {
                hr[r][x] = pack2(__uint_as_float(va[r * 16 + 2 * x]), __uint_as_float(va[r * 16 + 2 * x + 1]));
                hr[2 + r][x] = pack2(__uint_as_float(vb[r * 16 + 2 * x]), __uint_as_float(vb[r * 16 + 2 * x + 1]));
              }
          }
          if (half == 1) {                         // both halves of the accumulator are in registers / staged
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tm_empty[ts]);
          }
          // level 0: the thread's 4 patch rows x 16 columns = four adjacent 4x4 tiles = one 128-byte run
          unsigned char* sp = slot + half * 128;
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            *reinterpret_cast<uint4*>(sp + t * 32) = make_uint4(hr[0][2 * t], hr[0][2 * t + 1], hr[1][2 * t], hr[1][2 * t + 1]);
            *reinterpret_cast<uint4*>(sp + t * 32 + 16) = make_uint4(hr[2][2 * t], hr[2][2 * t + 1], hr[3][2 * t], hr[3][2 * t + 1]);
          }
          // pooled levels go to the band pool: wait (once per band) until its previous content has left
          if (!pool_ok) { mbar_wait(band_empty, (band & 1) ^ 1); pool_ok = true; }
          uint32_t l1[2][4];
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              l1[cc][j] = pack2(pool_pair(hr[2 * cc][2 * j], hr[2 * cc + 1][2 * j]),
                                pool_pair(hr[2 * cc][2 * j + 1], hr[2 * cc + 1][2 * j + 1]));
            unsigned char* st = pool1 + row * p1src + (2 * half + cc) * 8;
            *reinterpret_cast<uint2*>(st + (xb * 2) * 32) = make_uint2(l1[cc][0], l1[cc][1]);
            *reinterpret_cast<uint2*>(st + (xb * 2 + 1) * 32) = make_uint2(l1[cc][2], l1[cc][3]);
          }
          const uint32_t a0 = pack2(pool_pair(l1[0][0], l1[1][0]), pool_pair(l1[0][1], l1[1][1]));
          const uint32_t a1 = pack2(pool_pair(l1[0][2], l1[1][2]), pool_pair(l1[0][3], l1[1][3]));
          *reinterpret_cast<uint2*>(pool2 + row * p2src + half * p2row + xb * 8) = make_uint2(a0, a1);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&st_full[ts]);
        tph ^= 1; sph ^= 1;
      }
      if (!pool_ok) mbar_wait(band_empty, (band & 1) ^ 1);     // (a group without a tile in this band)
      __syncwarp();
      if (lane == 0) mbar_arrive(band_full);       // this warp's part of the band pool is complete
    }
  } else {
    // ===================== store warps =====================
    // One STG.256 instruction = 8 source pixels x one whole 128-byte run (lane -> pixel lane/4, 32-byte piece lane%4):
    // 8 LSU wavefronts of 128 B instead of the 32 wavefronts of 32 B a thread-per-pixel mapping costs.  (ncu, round 2:
    // l1tex__data_pipe_lsu_wavefronts was the top unit at 77-80 %.)
    const int row = threadIdx.x - (64 + kDrainWarps * 32);       // 0..127
    const int swarp = row >> 5;
    const int sub = lane >> 2, piece = lane & 3;
    int tile = 0, band = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++band) {
      const int yb = item % p.n_yb;
      const int mt = (item / p.n_yb) % p.n_mt;
      const int n = item / (p.n_yb * p.n_mt);
      const int n_out = p.out_slot ? __ldg(p.out_slot + n) : n;
      const long long pl0 = (long long)n_out * p.hw + mt * kBM;       // plane of the tile's first source pixel
      const int n_src = min(kBM, p.hw - mt * kBM);                    // valid source pixels of this tile
      for (int xb = 0; xb < p.n_xb; ++xb, ++tile) {
        const int s_ = tile & (kTStages - 1);
        mbar_wait(&st_full[s_], (tile / kTStages) & 1);
        const bool col_ok = xb * 4 + piece < p.w4_0;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const int ty = 2 * yb + hf;
          uint4 va[4], vb[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const unsigned char* sp = smStage + s_ * kStageBytes + (swarp * 32 + g * 8 + sub) * kStageRow + hf * 128 + piece * 32;
            va[g] = *reinterpret_cast<const uint4*>(sp);
            vb[g] = *reinterpret_cast<const uint4*>(sp + 16);
          }
          if (ty < p.h4_0 && col_ok) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const int sr = swarp * 32 + g * 8 + sub;
              if (sr < n_src) {
                unsigned char* dst = reinterpret_cast<unsigned char*>(p.lvl[0]) +
                                     (((pl0 + sr) * p.h4_0 + ty) * p.w4_0 + xb * 4 + piece) * 32LL;
                asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "r"(va[g].x), "r"(va[g].y),
                             "r"(va[g].z), "r"(va[g].w), "r"(vb[g].x), "r"(vb[g].y), "r"(vb[g].z), "r"(vb[g].w) : "memory");
              }
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&st_empty[s_]);
      }
      // ---- band write-out: levels 1-3, staged byte-for-byte as they go to memory; consecutive lanes take consecutive
      // 32-byte sectors of one source pixel's piece, so a wavefront carries up to 128 B here too
      mbar_wait(band_full, band & 1);
      if (p.num_levels > 1) {
        if (yb < p.h4_1) {
          for (int idx = row; idx < n_src * p.w4_1; idx += kStoreWarps * 32) {
            const int sr = idx / p.w4_1, sec = idx - sr * p.w4_1;
            const unsigned char* sp1 = pool1 + sr * p1src + sec * 32;
            const uint4 a = *reinterpret_cast<const uint4*>(sp1), b = *reinterpret_cast<const uint4*>(sp1 + 16);
            unsigned char* g1 = reinterpret_cast<unsigned char*>(p.lvl[1]) + (((pl0 + sr) * p.h4_1 + yb) * p.w4_1 + sec) * 32LL;
            asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g1), "r"(a.x), "r"(a.y), "r"(a.z),
                         "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
          }
        }
        if (p.num_levels > 2 && 2 * yb < h2) {
          const int spp = p.pitch2 >> 5;                       // sectors per (source pixel, band) piece
          for (int idx = row; idx < n_src * spp; idx += kStoreWarps * 32) {
            const int sr = idx / spp, sec = idx - sr * spp;
            const unsigned char* sp2 = pool2 + sr * p2src + sec * 32;
            uint32_t rr[8];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint2 t = *reinterpret_cast<const uint2*>(sp2 + 8 * k);
              rr[2 * k] = t.x; rr[2 * k + 1] = t.y;
            }
            unsigned char* g2 = reinterpret_cast<unsigned char*>(p.lvl[2]) + ((pl0 + sr) * p.n_yb + yb) * (long long)p.pitch2 + sec * 32;
            asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g2), "r"(rr[0]), "r"(rr[1]), "r"(rr[2]),
                         "r"(rr[3]), "r"(rr[4]), "r"(rr[5]), "r"(rr[6]), "r"(rr[7]) : "memory");
          }
        }
        if (p.num_levels > 3 && yb < h3 && row < n_src) {
          const unsigned char* sp2 = pool2 + row * p2src;
          uint32_t rr[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) {                    // level-3 columns 2k, 2k+1 of this band's row
            rr[k] = 0u;
            if (k < p.n_xb) {
              const uint32_t t = *reinterpret_cast<const uint32_t*>(sp2 + 8 * k);
              const uint32_t t2 = *reinterpret_cast<const uint32_t*>(sp2 + 8 * k + 4);
              const uint32_t b = *reinterpret_cast<const uint32_t*>(sp2 + p2row + 8 * k);
              const uint32_t b2 = *reinterpret_cast<const uint32_t*>(sp2 + p2row + 8 * k + 4);
              rr[k] = pack2(pool_pair(t, b), pool_pair(t2, b2));
            }
          }
          unsigned char* g3 = reinterpret_cast<unsigned char*>(p.lvl[3]) + ((pl0 + row) * p.n_yb + yb) * 32LL;
          asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(g3), "r"(rr[0]), "r"(rr[1]), "r"(rr[2]),
                       "r"(rr[3]), "r"(rr[4]), "r"(rr[5]), "r"(rr[6]), "r"(rr[7]) : "memory");
        }
      }
      // the pool is read by all four store warps: hand it back only when every one of them is done with it
      __syncwarp();
      if (lane == 0) mbar_arrive(band_empty);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kTStages * kBN);
}

// [F, D, hw] (channel-major) -> [F, hw, D] (K-major), D = 128, times 1/4 in half — the reference's
// `fmap / 4.0` on the half tensor (src/modules/corr.py:71-72): exact for normal values.
__global__ void __launch_bounds__(256)
to_kmajor_kernel(const __half* __restrict__ in, __half* __restrict__ out, int hw) {
  __shared__ __align__(16) __half tile[kD][64 + 2];
  const int n = blockIdx.y;
  const int p0 = blockIdx.x * 64;
  const __half* src = in + (size_t)n * kD * hw;
  const __half q = __float2half_rn(0.25f);
  if ((hw & 7) == 0 && p0 + 64 <= hw) {
    // 16-byte loads (8 pixels of one channel), scaled as half2, stored as 4 words
    const __half2 q2 = __half2half2(q);
    for (int idx = threadIdx.x; idx < kD * 8; idx += 256) {
      const int k = idx >> 3, pp = (idx & 7) * 8;
      uint4 v = __ldg(reinterpret_cast<const uint4*>(src + (size_t)k * hw + p0 + pp));
      __half2* h = reinterpret_cast<__half2*>(&v);
      uint32_t* dstw = reinterpret_cast<uint32_t*>(&tile[k][pp]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const __half2 r = __hmul2(h[u], q2);
        dstw[u] = *reinterpret_cast<const uint32_t*>(&r);
      }
    }
  } else {
    for (int idx = threadIdx.x; idx < kD * 64; idx += 256) {
      const int k = idx / 64, pp = idx % 64;
      tile[k][pp] = (p0 + pp < hw) ? __hmul(src[(size_t)k * hw + p0 + pp], q) : __half(0.f);
    }
  }
  __syncthreads();
  __half* dst = out + ((size_t)n * hw + p0) * kD;
  for (int idx = threadIdx.x; idx < 64 * (kD / 2); idx += 256) {
    const int pp = idx / (kD / 2), k2 = idx % (kD / 2);
    if (p0 + pp < hw) {
      __half2 v = __halves2half2(tile[2 * k2][pp], tile[2 * k2 + 1][pp]);
      reinterpret_cast<__half2*>(dst + (size_t)pp * kD)[k2] = v;
    }
  }
}

constexpr int kSmemStagedMax = 227 * 1024 - 1024;

// Tensor maps depend only on (base pointer, frame count, h, w): a factor graph builds from the same video-level K-major
// buffer for its whole life, so the two encodes per launch are paid once.
enum { kMapA = 0, kMapB = 1 };

bool encode_map(GsEncodeTiledFn enc, const GsMapKey& k, CUtensorMap* out) {
  const int F = k.dims[0], h = k.dims[1], w = k.dims[2];
  const cuuint64_t hw = (cuuint64_t)h * w;
  if (k.kind == kMapA) {       // A: [F, hw, 128] as (ch, pixel, frame), box 64 ch x 128 pixels
    cuuint64_t dims[3] = {(cuuint64_t)kD, hw, (cuuint64_t)F};
    cuuint64_t strides[2] = {(cuuint64_t)kD * 2, hw * kD * 2};
    cuuint32_t box[3] = {(cuuint32_t)kKBox, (cuuint32_t)kBM, 1};
    cuuint32_t es[3] = {1, 1, 1};
    return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(k.base), dims, strides, box, es,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  // B: (ch, x, y, frame), box 64 ch x 16 x 8: an image patch; rows / columns outside the image read as zero
  cuuint64_t dims[4] = {(cuuint64_t)kD, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)F};
  cuuint64_t strides[3] = {(cuuint64_t)kD * 2, (cuuint64_t)w * kD * 2, hw * kD * 2};
  cuuint32_t box[4] = {(cuuint32_t)kKBox, (cuuint32_t)kPX, (cuuint32_t)kPY, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(k.base), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

GsMapCache g_maps(16, encode_map);
GsDeviceOnce g_device_once;

cudaError_t device_init(int) {
  cudaError_t e = cudaFuncSetAttribute(corr_build_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemTC);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(corr_build_tc_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemStagedMax);
  return e;
}

// launch the tensor-core kernel on K-major (pre-scaled) operands: f1t/f2t = [F1|F2, hw, 128]
int launch_tc(const __half* f1t, int F1, const __half* f2t, int F2, const int64_t* ii,
              const int64_t* jj, int rig, const int* out_slot, int tiled, __half* const* levels,
              int num_levels, int N, int h, int w, cudaStream_t st) {
  const int hw = h * w;
  CUtensorMap mapA, mapB;
  if (!g_maps.get(GsMapKey{f1t, kMapA, {F1, h, w}}, &mapA) || !g_maps.get(GsMapKey{f2t, kMapB, {F2, h, w}}, &mapB))
    return GOSLAM_ELAUNCH;
  const int rc = gs_device_once(g_device_once, device_init);
  if (rc != GOSLAM_OK) return rc;
  TcParams p{};
  for (int i = 0; i < 4; ++i) p.lvl[i] = i < num_levels ? levels[i] : nullptr;
  p.num_levels = num_levels; p.N = N; p.h = h; p.w = w; p.hw = hw;
  p.n_mt = gs_cdiv(hw, kBM); p.n_yb = gs_cdiv(h, kPY); p.n_xb = gs_cdiv(w, kPX);
  p.n_items = N * p.n_mt * p.n_yb;
  p.ii = ii; p.jj = jj; p.rig = rig; p.out_slot = out_slot;
  p.tiled = tiled ? 1 : 0;
  p.w4_0 = gs_cdiv(w, 4); p.h4_0 = gs_cdiv(h, 4);
  p.w4_1 = gs_cdiv(w >> 1, 4); p.h4_1 = gs_cdiv(h >> 1, 4);
  p.pitch2 = (p.n_xb * 16 + 31) / 32 * 32; p.pitch3 = 32;
  p.aligned = (w % 16 == 0 && h % 8 == 0) ? 1 : 0;
  const int sms = gs_sm_count();
  const int grid = p.n_items < sms ? p.n_items : sms;
  if (p.tiled && p.num_levels == 4 && smem_staged(p.n_xb) <= kSmemStagedMax) {
    corr_build_tc_staged_kernel<<<grid, kThreadsST, smem_staged(p.n_xb), st>>>(mapA, mapB, p, pool_bytes_st(p.n_xb));
    GS_CHECK_LAUNCH();
    return GOSLAM_OK;
  }
  corr_build_tc_kernel<<<grid, kThreadsTC, kSmemTC, st>>>(mapA, mapB, p);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int build_tc(const __half* f1, const __half* f2, __half* const* levels, int num_levels, int N,
             int h, int w, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  const int hw = h * w;
  const size_t per = (size_t)N * hw * kD * sizeof(__half);
  if (workspace == nullptr || workspace_bytes < 2 * gs_align(per)) return GOSLAM_EWORKSPACE;
  __half* f1t = reinterpret_cast<__half*>(workspace);
  __half* f2t = reinterpret_cast<__half*>(reinterpret_cast<char*>(workspace) + gs_align(per));
  dim3 tg(gs_cdiv(hw, 64), N);
  to_kmajor_kernel<<<tg, 256, 0, st>>>(f1, f1t, hw);
  to_kmajor_kernel<<<tg, 256, 0, st>>>(f2, f2t, hw);
  GS_CHECK_LAUNCH();
  return launch_tc(f1t, N, f2t, N, nullptr, nullptr, 1, nullptr, 0, levels, num_levels, N, h, w, st);
}

}  // namespace

extern "C" {

size_t goslam_corr_build_workspace_bytes(int N, int D, int h, int w) {
  if (N <= 0 || D != kD) return 256;
  return 2 * gs_align((size_t)N * h * w * kD * sizeof(__half)) + 256;
}

int goslam_fmaps_to_kmajor(const void* fmaps, void* out, int F, int D, int h, int w, void* stream) {
  if (F < 0 || D != kD || h <= 0 || w <= 0) return GOSLAM_EINVAL;
  if (F == 0) return GOSLAM_OK;
  dim3 tg(gs_cdiv(h * w, 64), F);
  to_kmajor_kernel<<<tg, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __half*>(fmaps),
                                                         reinterpret_cast<__half*>(out), h * w);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int goslam_corr_build_indexed(const void* fmaps_kmajor, int F, int rig, const int64_t* ii,
                              const int64_t* jj, void* const* levels, int num_levels, int N, int D,
                              int h, int w, void* stream) {
  return goslam_corr_pool_build(fmaps_kmajor, F, rig, ii, jj, nullptr, GOSLAM_LAYOUT_ROWMAJOR, levels,
                                num_levels, N, D, h, w, stream);
}

size_t goslam_corr_level_plane_elems(int level, int layout, int h, int w) {
  if (level < 0 || level > 3 || h <= 0 || w <= 0) return 0;
  const int hl = h >> level, wl = w >> level;
  if (hl <= 0 || wl <= 0) return 0;
  if (layout == GOSLAM_LAYOUT_TILED) {
    if (level < 2) return (size_t)gs_cdiv(hl, 4) * gs_cdiv(wl, 4) * 16;
    // levels 2 / 3: one padded piece per 8-row band of level 0 (2 rows / 1 row of the level)
    const int n_yb = gs_cdiv(h, kPY), n_xb = gs_cdiv(w, kPX);
    return level == 2 ? (size_t)n_yb * ((n_xb * 8 + 15) / 16 * 16) : (size_t)n_yb * 16;
  }
  return (size_t)hl * wl;
}

int goslam_corr_pool_build(const void* fmaps_kmajor, int F, int rig, const int64_t* ii,
                           const int64_t* jj, const int* slots, int layout, void* const* levels,
                           int num_levels, int N, int D, int h, int w, void* stream) {
  if (layout != GOSLAM_LAYOUT_ROWMAJOR && layout != GOSLAM_LAYOUT_TILED) return GOSLAM_EINVAL;
  if (N < 0 || F <= 0 || rig < 1 || D != kD || h <= 0 || w <= 0 || num_levels < 1 || num_levels > 4)
    return GOSLAM_EINVAL;
  if ((h >> (num_levels - 1)) <= 0 || (w >> (num_levels - 1)) <= 0) return GOSLAM_EINVAL;
  if (w > kMaxXB * kPX) return GOSLAM_EINVAL;
  if (N == 0) return GOSLAM_OK;
  const __half* f = reinterpret_cast<const __half*>(fmaps_kmajor);
  return launch_tc(f, F, f, F, ii, jj, rig, slots, layout == GOSLAM_LAYOUT_TILED,
                   reinterpret_cast<__half* const*>(levels), num_levels, N, h, w, (cudaStream_t)stream);
}

int goslam_corr_build(const void* fmap1, const void* fmap2, void* const* levels, int num_levels,
                      int N, int D, int h, int w, int impl, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (N < 0 || D <= 0 || h <= 0 || w <= 0 || num_levels < 1 || num_levels > 4) return GOSLAM_EINVAL;
  if ((h >> (num_levels - 1)) <= 0 || (w >> (num_levels - 1)) <= 0) return GOSLAM_EINVAL;
  if (N == 0) return GOSLAM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const __half* f1 = reinterpret_cast<const __half*>(fmap1);
  const __half* f2 = reinterpret_cast<const __half*>(fmap2);
  __half* const* lv = reinterpret_cast<__half* const*>(levels);
  if (impl == 0) impl = (D == kD && w <= kMaxXB * kPX) ? 1 : 2;
  if (impl == 1) {
    if (D != kD || w > kMaxXB * kPX) return GOSLAM_EINVAL;
    return build_tc(f1, f2, lv, num_levels, N, h, w, workspace, workspace_bytes, st);
  }
  if (impl == 2) return gs_corr_build_simt_f16(f1, f2, lv, num_levels, N, D, h, w, st);
  return GOSLAM_EINVAL;
}

}  // extern "C"
