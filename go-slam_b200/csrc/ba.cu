// ba.cu — dense Gauss-Newton bundle adjustment over SE3 poses x per-pixel inverse depth.
//
// Replaces droid_backends.ba = ba_cuda (src/lib/droid_kernels.cu:1314-1434) together with
// projective_transform_kernel (:176-424), accum_kernel/accum_cuda (:854-998), EEt6x6 /
// Ev6x1 / EvT6x1 (:1001-1115), pose/disp retraction (:898-946) and the host-side Eigen
// pose-block assembly + Schur complement + SimplicialLLT (:1117-1311).
//
// What is different from the reference (same mathematics, same constants, same quirks):
//   * NOTHING leaves the device: the frame set (`torch::_unique`), the edge->frame CSR that
//     accum_cuda rebuilds on the CPU four times per iteration, the Schur pair list that
//     schur_block builds with O(P^2 deg^2) host loops, and the float64 LLT all run in
//     kernels; zero D2H/H2D copies and zero host synchronisation per call.
//   * Linearisation is FRAME-major (one thread = one pixel of a source keyframe, looping
//     over that keyframe's outgoing edges) so the per-pixel depth Hessian C, the depth
//     gradient w, Q = 1/C and E_i = sum_e E_ii are complete in registers when the loop ends
//     — no accum passes over [N,hw] temporaries.
//   * J_i = -Ad^T J_j is linear, so only H_jj (21) and v_j (6) are reduced per edge (a
//     27-value warp transpose-reduction, 31 shuffles instead of 90 block reductions);
//     H_ii, H_ij, v_i follow from a 6x6 adjoint sandwich in the assembly step, in float64.
//   * The reduced camera system is accumulated and solved in float64 on the device
//     (the reference converts fp32 blocks to float64 and solves on the CPU).
//
//   * Small windows (6P <= 96, every local window): ALL Gauss-Newton iterations of a call run in
//     ONE cooperative kernel (ba_persistent_kernel) — linearise | grid barrier | reduced system |
//     grid barrier | solve (block 0) | grid barrier, with the depth back-substitution of iteration
//     i fused into the linearisation of iteration i+1; larger systems and the multi-GPU split
//     form (goslam_ba_phase1/2) run the same device functions as separate launches.
//
// Reference quirks kept on purpose: the first optimised pose is skipped in the depth
// back-substitution (`ix <= 0`, :1105); C/b_z use the stereo edge's weight before it is
// zeroed (:320-323); stereo baseline (-0.1,0,0) (:219-229); MIN_DEPTH 0.25 (:26);
// damping diag += ep + lm*diag (:1197); failed factorisation => dx = 0 (:1207-1210).
#include "common.cuh"
#include "launch.cuh"
#include <cstring>
#include "se3.cuh"
#include <algorithm>
#include <cstdio>
#include <cooperative_groups.h>

namespace {

constexpr int kTP = 128;       // pixels (threads) per linearise / back-substitute block
constexpr int kNRed = 27;      // 21 (H_jj upper) + 6 (v_j)
constexpr float kAlpha = 0.05f;  // sensor-depth prior weight (src/lib/droid_kernels.cu:1396)

struct BaWs {
  // graph tables (built once per call by ba_prep_kernel)
  int* slot_of_frame;  // [num]   slot in kx or -1
  int* kx;             // [num]   frame id of slot
  int* counts;         // [8]     M, total_entries, total_pairs, grid-barrier counter, bad-argument flag
  int* row_ptr;        // [num+1] CSR over frame id: edges with ii == frame
  int* edge_idx;       // [N]
  int* entry_ptr;      // [num+1] per slot: Schur entries
  int* entry_code;     // [num+N] >=0: edge id (E_ij), <0: -(pose+1) (E_i of that pose)
  int* pair_ptr;       // [num+1] per slot: prefix of ne*(ne+1)/2
  int* edge_j;         // [N]     jj as int (kept for the split phase-2 entry point)
  // per-iteration buffers
  float* Eij;          // [N,6,hw]
  float* Ei;           // [num(slot),6,hw]
  float* Q;            // [num(slot),hw]
  float* w;            // [num(slot),hw]
  float* part;         // [N,ntiles*kTP/32,27]  one partial per (edge, tile, warp)
  double* sys;         // [n*n + n]  reduced camera system (H row-major, then b)
  double* chol;        // [n*n]      factor scratch (global path)
  double* rhs;         // [n]        rhs / solution scratch (global path)
  float* dx;           // [P,6]
  int ntiles;
};

struct BaDims {
  int N, num, ht, wd, hw, t0, t1, P, n;
};

size_t ba_layout(const BaDims& d, void* base, size_t cap, BaWs* ws) {
  GsArena a(base, cap);
  const int ntiles = gs_cdiv(d.hw, kTP);
  BaWs w{};
  w.slot_of_frame = a.take<int>(d.num);
  w.kx = a.take<int>(d.num);
  w.counts = a.take<int>(8);
  w.row_ptr = a.take<int>(d.num + 1);
  w.edge_idx = a.take<int>(d.N > 0 ? d.N : 1);
  w.entry_ptr = a.take<int>(d.num + 1);
  w.entry_code = a.take<int>(d.num + d.N);
  w.pair_ptr = a.take<int>(d.num + 1);
  w.edge_j = a.take<int>(d.N > 0 ? d.N : 1);
  w.Eij = a.take<float>((size_t)(d.N > 0 ? d.N : 1) * 6 * d.hw);
  w.Ei = a.take<float>((size_t)d.num * 6 * d.hw);
  w.Q = a.take<float>((size_t)d.num * d.hw);
  w.w = a.take<float>((size_t)d.num * d.hw);
  w.part = a.take<float>((size_t)(d.N > 0 ? d.N : 1) * ntiles * (kTP / 32) * kNRed);
  w.sys = a.take<double>((size_t)d.n * d.n + d.n);
  w.chol = a.take<double>((size_t)d.n * d.n);
  w.rhs = a.take<double>(d.n > 0 ? d.n : 1);
  w.dx = a.take<float>((size_t)(d.P > 0 ? d.P : 1) * 6);
  w.ntiles = ntiles;
  if (ws) *ws = w;
  return a.off;
}

// ------------------------------------------------------------------------------------
// Graph tables.  One block; everything is indexed by frame id so "sorted unique" is a
// prefix sum over a presence bitmap (frame order == sorted order, as torch::_unique gives).
// All prefix sums are block-wide scans (warp shuffles + one shared-memory hop), the per-frame
// degree is counted with shared-memory atomics, the CSR keeps the edges of a frame in edge-index
// order (stable: the linearisation's summation order does not depend on thread scheduling).
// Round 1 did the scans and the Schur tables in thread 0 (chains of dependent global loads).
// ------------------------------------------------------------------------------------
constexpr int kPrepThreads = 1024;
constexpr int kPrepMaxFrames = 4 * kPrepThreads;       // == the 4096 of make_dims

// in-place exclusive scan of a[0..n) in shared memory, n <= 4 * blockDim.x; returns the total.  All threads call.
__device__ int prep_excl_scan(int* a, int n, int* wsum /* [33] */) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int per = (n + (int)blockDim.x - 1) / (int)blockDim.x;
  const int base = tid * per;
  int loc[4], s = 0;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    loc[q] = s;
    if (q < per && base + q < n) s += a[base + q];
  }
  int inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int w = lane < ((int)blockDim.x >> 5) ? wsum[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    wsum[lane] = winc - w;
    if (lane == 31) wsum[32] = winc;
  }
  __syncthreads();
  const int off = wsum[warp] + inc - s;
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (q < per && base + q < n) a[base + q] = off + loc[q];
  const int total = wsum[32];
  __syncthreads();
  return total;
}

__global__ void __launch_bounds__(kPrepThreads)
ba_prep_kernel(const int64_t* __restrict__ ii, const int64_t* __restrict__ jj, BaDims d, BaWs ws, int zero,
               int eta_rows) {
  extern __shared__ int sm[];          // a[num] | b[num + 1] | c[num] | wsum[33]
  const int tid = threadIdx.x, nt = blockDim.x;
  if (zero) {                          // single-kernel driver: reduced system and grid-barrier counter start at 0
    const size_t nsys = (size_t)d.n * d.n + d.n;
    for (size_t i = tid; i < nsys; i += nt) ws.sys[i] = 0.0;
    if (tid == 0) ws.counts[3] = 0;
  }
  int* a = sm;                         // presence -> entries per slot -> entry_ptr
  int* b = sm + d.num;                 // degree -> row_ptr (kept)
  int* c = b + d.num + 1;              // slot scan -> pairs per slot -> pair_ptr
  int* wsum = c + d.num;
  for (int f = tid; f < d.num; f += nt) { a[f] = (f >= d.t0 && f < d.t1) ? 1 : 0; b[f] = 0; }
  __syncthreads();
  for (int e = tid; e < d.N; e += nt) {
    const int f = (int)ii[e];
    if (f >= 0 && f < d.num) { a[f] = 1; atomicAdd(&b[f], 1); }     // presence: benign race, all write 1
    ws.edge_j[e] = (int)jj[e];
  }
  __syncthreads();
  // ---- depth slots: frames of [t0,t1) U ii in sorted order ----
  for (int f = tid; f < d.num; f += nt) c[f] = a[f];
  __syncthreads();
  const int M = prep_excl_scan(c, d.num, wsum);
  for (int f = tid; f < d.num; f += nt) {
    if (a[f]) { ws.slot_of_frame[f] = c[f]; ws.kx[c[f]] = f; }
    else ws.slot_of_frame[f] = -1;
  }
  if (tid == 0) {
    ws.counts[0] = M;
    // eta must have one row (broadcast), one row per depth slot (the reference's
    // `damping[unique(cat(arange(t0,t1), ii))]`, src/factor_graph.py:236-238) or — negative
    // eta_rows — one row per FRAME.  Anything else is a caller bug that the reference reports as a
    // broadcast error (src/lib/droid_kernels.cu:1397); here the call becomes a no-op with status 2.
    ws.counts[4] = (eta_rows == 0 || eta_rows == 1 || eta_rows == M || eta_rows == -d.num) ? 0 : 1;
  }
  // ---- CSR over source frames, edges of a frame in edge-index order ----
  const int n_listed = prep_excl_scan(b, d.num, wsum);
  if (tid == 0) b[d.num] = n_listed;
  __syncthreads();
  for (int f = tid; f <= d.num; f += nt) ws.row_ptr[f] = b[f];
  for (int e = tid; e < d.N; e += nt) {
    const int f = (int)ii[e];
    if (f < 0 || f >= d.num) continue;
    int rank = 0;
    for (int q = 0; q < e; ++q) rank += ((int)ii[q] == f);          // stable position inside the frame's run
    ws.edge_idx[b[f] + rank] = e;
  }
  __syncthreads();                     // edge_idx (global) is read below by other threads of this block
  // ---- Schur entries per slot: [E_i of the frame's own pose if optimised] + [E_ij of each outgoing edge whose
  // target pose is optimised]  (schur_block graph, :1244-1253); pairs = ne (ne + 1) / 2 ----
  for (int k = tid; k < d.num; k += nt) {
    int ne = 0;
    if (k < M) {
      const int f = ws.kx[k];            // written by another thread of this block, visible after the barriers above
      ne = (f >= d.t0 && f < d.t1) ? 1 : 0;
      for (int r = b[f]; r < b[f + 1]; ++r) {
        const int j = (int)jj[ws.edge_idx[r]];
        ne += (j >= d.t0 && j < d.t1) ? 1 : 0;
      }
    }
    // (a and c are dead as presence / slot index from here on: their last readers are behind a barrier)
    a[k] = ne;
    c[k] = ne * (ne + 1) / 2;
  }
  __syncthreads();
  const int n_entries = prep_excl_scan(a, d.num, wsum);
  const int n_pairs = prep_excl_scan(c, d.num, wsum);
  for (int k = tid; k < M; k += nt) {
    const int f = ws.kx[k];
    int eo = a[k];
    ws.entry_ptr[k] = eo;
    ws.pair_ptr[k] = c[k];
    if (f >= d.t0 && f < d.t1) ws.entry_code[eo++] = -(f - d.t0 + 1);
    for (int r = b[f]; r < b[f + 1]; ++r) {
      const int e = ws.edge_idx[r];
      const int j = (int)jj[e];
      if (j >= d.t0 && j < d.t1) ws.entry_code[eo++] = e;
    }
  }
  if (tid == 0) {
    ws.entry_ptr[M] = n_entries;
    ws.pair_ptr[M] = n_pairs;
    ws.counts[1] = n_entries;
    ws.counts[2] = n_pairs;
  }
}

// 32 values per lane -> lane L returns sum over lanes of v[L]   (31 shuffles)
__device__ __forceinline__ float warp_transpose_reduce32(float (&v)[32], int lane) {
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

// ------------------------------------------------------------------------------------
// Linearise: grid (ntiles, num); block = kTP pixels of slot blockIdx.y.
// ------------------------------------------------------------------------------------
struct BaIn {
  const float* poses; const float* disps; const float* intr; const float* disps_sens;
  const float* targets; const float* weights; const float* eta; int eta_rows;
  const int64_t* ii; const int64_t* jj;
};

// One (frame slot k, kTP-pixel tile) unit; blockDim.x == kTP.  poses / disps are deliberately
// NOT __restrict__: the single-kernel path below rewrites them between iterations.
__device__ __forceinline__ void linearize_tile(const BaIn& in, const BaDims& d, const BaWs& ws,
                                               int motion_only, int k, int wt) {
  const float* poses = in.poses; const float* disps = in.disps;
  const float* __restrict__ intr = in.intr; const float* __restrict__ disps_sens = in.disps_sens;
  const float* __restrict__ targets = in.targets; const float* __restrict__ weights = in.weights;
  const float* __restrict__ eta = in.eta; const int eta_rows = in.eta_rows;
  const int f = ws.kx[k];
  // wt = 32-pixel warp tile of the frame (no block-level cooperation anywhere below)
  const int lane = threadIdx.x & 31;
  const int px = wt * 32 + lane;
  const bool act = px < d.hw;

  const float fx = intr[0], fy = intr[1], cx = intr[2], cy = intr[3];
  const float u = (float)(px % d.wd), v = (float)(px / d.wd);
  const float di = act ? disps[(size_t)f * d.hw + px] : 1.0f;
  float Xi[4] = {(u - cx) / fx, (v - cy) / fy, 1.0f, di};

  float C = 0.f, wz = 0.f;
  float Ei[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};

  const int r0 = ws.row_ptr[f], r1 = ws.row_ptr[f + 1];
  // Software pipeline over the frame's edges (the loop is a chain of dependent look-ups otherwise:
  // edge id -> target frame -> pose): the edge id / target frame are fetched two edges ahead, the
  // target pose and the pixel's target / weight one edge ahead.
  float pi[7];
#pragma unroll
  for (int c = 0; c < 7; ++c) pi[c] = poses[7 * (size_t)f + c];
  int e1 = 0, j1 = f, e2 = 0, j2 = f;                  // edge r (then r+1) and edge r+1 (then r+2)
  if (r0 < r1) { e1 = ws.edge_idx[r0]; j1 = ws.edge_j[e1]; }
  if (r0 + 1 < r1) { e2 = ws.edge_idx[r0 + 1]; j2 = ws.edge_j[e2]; }
  float nx[4] = {0.f, 0.f, 0.f, 0.f}, pn[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f};
  if (r0 < r1) {
    if (act) {
      const size_t o = ((size_t)e1 * 2) * d.hw + px;
      nx[0] = targets[o]; nx[1] = targets[o + d.hw]; nx[2] = weights[o]; nx[3] = weights[o + d.hw];
    }
#pragma unroll
    for (int c = 0; c < 7; ++c) pn[c] = poses[7 * (size_t)j1 + c];
  }
  for (int r = r0; r < r1; ++r) {
    const int e = e1, jx = j1;
    const float tu = nx[0], tv = nx[1], qu = nx[2], qv = nx[3];
    float pj[7];
#pragma unroll
    for (int c = 0; c < 7; ++c) pj[c] = pn[c];
    e1 = e2; j1 = j2;
    if (r + 1 < r1) {
      if (act) {
        const size_t o = ((size_t)e1 * 2) * d.hw + px;
        nx[0] = targets[o]; nx[1] = targets[o + d.hw]; nx[2] = weights[o]; nx[3] = weights[o + d.hw];
      }
#pragma unroll
      for (int c = 0; c < 7; ++c) pn[c] = poses[7 * (size_t)j1 + c];
    }
    if (r + 2 < r1) { e2 = ws.edge_idx[r + 2]; j2 = ws.edge_j[e2]; }
    const bool stereo = (jx == f);
    GsSE3 G;
    if (stereo) {                                     // fixed stereo baseline (see gs_edge_pose)
      G.t[0] = -0.1f; G.t[1] = 0.f; G.t[2] = 0.f;
      G.q[0] = 0.f; G.q[1] = 0.f; G.q[2] = 0.f; G.q[3] = 1.f;
    } else {
      gs_rel(pi, pi + 3, pj, pj + 3, G);
    }

    float Xj[4];
    gs_act4(G, Xi, Xj);
    const float x = Xj[0], y = Xj[1], h = Xj[3];
    const bool behind = Xj[2] < GS_MIN_DEPTH;
    // reference: d = 1.0 / Xj[2] in double, then narrowed to float.  RN_f32(RN_f64(1/Z)) equals the
    // correctly rounded float reciprocal unless the double quotient lands within 2^-53 of a float
    // rounding midpoint (impossible exactly, since 1/Z has no finite midpoint expansion) — so the
    // single-instruction float reciprocal is used instead of an fp64 divide.
    const float dd = behind ? 0.0f : __frcp_rn(Xj[2]);
    const float d2 = dd * dd;
    float wu = (behind || !act) ? 0.0f : (float)(.001 * (double)qu);
    float wv = (behind || !act) ? 0.0f : (float)(.001 * (double)qv);
    const float ru = tu - (fx * dd * x + cx);
    const float rv = tv - (fy * dd * y + cy);

    float Ju[6], Jv[6];
    Ju[0] = fx * (h * dd);       Ju[1] = fx * 0.f;
    Ju[2] = fx * (-x * h * d2);  Ju[3] = fx * (-x * y * d2);
    Ju[4] = fx * (1 + x * x * d2);  Ju[5] = fx * (-y * dd);
    Jv[0] = fy * 0.f;            Jv[1] = fy * (h * dd);
    Jv[2] = fy * (-y * h * d2);  Jv[3] = fy * (-1 - y * y * d2);
    Jv[4] = fy * (x * y * d2);   Jv[5] = fy * (x * dd);
    const float Jzu = fx * (G.t[0] * dd - G.t[2] * (x * d2));
    const float Jzv = fy * (G.t[1] * dd - G.t[2] * (y * d2));

    C += wu * Jzu * Jzu;  C += wv * Jzv * Jzv;
    wz += wu * ru * Jzu;  wz += wv * rv * Jzv;
    if (stereo) { wu = 0.f; wv = 0.f; }

    // H_jj (upper triangle, row-major) and v_j
    float val[32];
    {
      int l = 0;
#pragma unroll
      for (int a = 0; a < 6; ++a)
#pragma unroll
        for (int b = a; b < 6; ++b) val[l++] = wu * Ju[a] * Ju[b] + wv * Jv[a] * Jv[b];
#pragma unroll
      for (int a = 0; a < 6; ++a) val[21 + a] = wu * ru * Ju[a] + wv * rv * Jv[a];
#pragma unroll
      for (int a = kNRed; a < 32; ++a) val[a] = 0.f;
    }
    // one partial per warp: no block barrier anywhere in the linearisation
    const float tot = warp_transpose_reduce32(val, lane);
    if (lane < kNRed)
      ws.part[((size_t)e * ws.ntiles * (kTP / 32) + wt) * kNRed + lane] = tot;

    if (!motion_only) {
      float Ee[6], Eii[6];
#pragma unroll
      for (int a = 0; a < 6; ++a) Ee[a] = wu * Jzu * Ju[a] + wv * Jzv * Jv[a];
      gs_adjT(G, Ee, Eii);       // E_ii = -Ad^T E_ij
      if (act) {
#pragma unroll
        for (int a = 0; a < 6; ++a) {
          ws.Eij[((size_t)e * 6 + a) * d.hw + px] = Ee[a];
          Ei[a] -= Eii[a];
        }
      }
    }
  }

  if (!motion_only && act) {
    // depth prior where the sensor has a reading, eta-damping elsewhere (:1396-1400)
    const float ds = disps_sens[(size_t)f * d.hw + px];
    const float m = (ds > 0.f) ? 1.0f : 0.0f;
    const int er = (eta_rows == 1) ? 0 : (eta_rows < 0 ? f : k);
    const float et = eta[(size_t)er * d.hw + px];
    C = C + m * kAlpha + (1.0f - m) * et;
    wz = wz - m * kAlpha * (di - ds);
    const size_t o = (size_t)k * d.hw + px;
    ws.Q[o] = 1.0f / C;
    ws.w[o] = wz;
#pragma unroll
    for (int a = 0; a < 6; ++a) ws.Ei[((size_t)k * 6 + a) * d.hw + px] = Ei[a];
  }
}

__global__ void __launch_bounds__(kTP)
ba_linearize_kernel(BaIn in, BaDims d, BaWs ws, int motion_only) {
  if ((int)blockIdx.y >= ws.counts[0] || ws.counts[4]) return;
  linearize_tile(in, d, ws, motion_only, blockIdx.y, blockIdx.x * (kTP / 32) + (threadIdx.x >> 5));
}

// ------------------------------------------------------------------------------------
// Reduced camera system accumulation (persistent blocks):
//   items [0, N)            pose blocks of edge e from its H_jj/v_j partials (A, :1376-1383)
//   items [N, N + npairs)   Schur pair (a,b) of a depth frame: S_ab = sum_px E_a Q E_b^T,
//                           and for a == b also v_a = sum_px E_a Q w   (:1001-1093,:1257-1311)
// sys = (A - S | b_A - b_S) in float64.
// ------------------------------------------------------------------------------------
struct SysSmem {
  float red[8][64];
  double redd[8][32];
  double Hs[36], Ms[36], Ts[36], vs[6];
};

// items first, first + stride, ... ; NT threads per block (poses not __restrict__, see above)
template <int NT>
__device__ __forceinline__ void system_items(const float* poses, const int64_t* __restrict__ ii,
                                             const int64_t* __restrict__ jj, const BaDims& d,
                                             const BaWs& ws, int motion_only, int bid, int nb,
                                             SysSmem& sm) {
  float (*red)[64] = sm.red;
  double* Hs = sm.Hs; double* Ms = sm.Ms; double* Ts = sm.Ts; double* vs = sm.vs;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int M = ws.counts[0];
  const int npairs = motion_only ? 0 : ws.counts[2];
  constexpr int kChunk = 4 * NT;                     // pixels per Schur work unit (4 per thread)
  const int nchunk = (d.hw + kChunk - 1) / kChunk;
  double* H = ws.sys;
  double* bvec = ws.sys + (size_t)d.n * d.n;

  // ---------------- pose blocks of the edges ----------------
  // Edges go to the blocks at the END of the grid: the Schur ranges below fill it from the front
  // and usually leave the tail idle.
  for (int e = nb - 1 - bid; e < d.N; e += nb) {
    const int ix = (int)ii[e], jx = (int)jj[e];
    const int pi = ix - d.t0, pj = jx - d.t0;
    const bool vi_ok = pi >= 0 && pi < d.P, vj_ok = pj >= 0 && pj < d.P;
    if ((!vi_ok && !vj_ok) || ix < 0 || ix >= d.num) continue;
    // per-tile partials -> 27 sums: warp w takes tiles w, w + NT/32, ... (independent loads)
    {
      double ps = 0.0;
      if (lane < kNRed) {
        const int nparts = ws.ntiles * (kTP / 32);
        const float* pp = ws.part + (size_t)e * nparts * kNRed + lane;
#pragma unroll 8
        for (int t = warp; t < nparts; t += NT / 32) ps += (double)pp[(size_t)t * kNRed];
      }
      sm.redd[warp][lane] = ps;
    }
    __syncthreads();
    if (tid < kNRed) {
      double s = 0.0;
#pragma unroll
      for (int wq = 0; wq < NT / 32; ++wq) s += sm.redd[wq][tid];
      if (tid < 21) {
        // unpack upper-triangular index -> (a,b)
        int a = 0, l = tid;
        while (l >= 6 - a) { l -= 6 - a; ++a; }
        const int b = a + l;
        Hs[a * 6 + b] = s; Hs[b * 6 + a] = s;
      } else {
        vs[tid - 21] = s;
      }
    }
    if (tid >= 32 && tid < 38) {
      // column c of M = Ad^T (apply the dual adjoint to unit vector c)
      const int c = tid - 32;
      GsSE3 G;
      gs_edge_pose(poses, ix, jx, G);
      float X[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, Y[6];
      X[c] = 1.0f;
      gs_adjT(G, X, Y);
      for (int r = 0; r < 6; ++r) Ms[r * 6 + c] = (double)Y[r];
    }
    __syncthreads();
    // T = M * Hjj
    if (tid < 36) {
      const int r = tid / 6, c = tid % 6;
      double s = 0.0;
      for (int q = 0; q < 6; ++q) s += Ms[r * 6 + q] * Hs[q * 6 + c];
      Ts[tid] = s;
    }
    __syncthreads();
    if (tid < 36) {
      const int r = tid / 6, c = tid % 6;
      // Hii = M Hjj M^T = T M^T ; Hij = -M Hjj = -T ; Hji = Hij^T ; vi = -M vj
      if (vi_ok) {
        double s = 0.0;
        for (int q = 0; q < 6; ++q) s += Ts[r * 6 + q] * Ms[c * 6 + q];
        atomicAdd(&H[(size_t)(6 * pi + r) * d.n + 6 * pi + c], s);
      }
      if (vi_ok && vj_ok) {
        atomicAdd(&H[(size_t)(6 * pi + r) * d.n + 6 * pj + c], -Ts[r * 6 + c]);
        atomicAdd(&H[(size_t)(6 * pj + r) * d.n + 6 * pi + c], -Ts[c * 6 + r]);
      }
      if (vj_ok) atomicAdd(&H[(size_t)(6 * pj + r) * d.n + 6 * pj + c], Hs[r * 6 + c]);
    } else if (tid >= 64 && tid < 70) {
      const int r = tid - 64;
      if (vj_ok) atomicAdd(&bvec[6 * pj + r], vs[r]);
      if (vi_ok) {
        double s = 0.0;
        for (int q = 0; q < 6; ++q) s += Ms[r * 6 + q] * vs[q];
        atomicAdd(&bvec[6 * pi + r], -s);
      }
    }
    __syncthreads();
  }

  // ---------------- Schur pairs ----------------
  // Work unit = (pair, 4*NT-pixel chunk); every block takes a CONTIGUOUS range of units, so it
  // mostly stays inside one pair: the pair is decoded once (a chain of dependent table look-ups)
  // and its 42 sums are reduced and flushed once, however many chunks the block adds to them.
  const int total = npairs * nchunk;
  const int per = (total + nb - 1) / nb;
  const int u0 = bid * per;
  const int u1 = min(total, u0 + per);
  int cur = -1, pa = 0, pb = 0;
  bool diag = false;
  const float* Ea = nullptr; const float* Eb = nullptr; const float* Qk = nullptr; const float* wk = nullptr;
  float acc[64];
  auto flush = [&]() {
    // two 32-wide transpose reductions: values [0,32) and [32,64)
    float lo32[32], hi32[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) { lo32[i] = acc[i]; hi32[i] = acc[32 + i]; }
    const float s0 = warp_transpose_reduce32(lo32, lane);
    const float s1 = warp_transpose_reduce32(hi32, lane);
    red[warp][lane] = s0;
    red[warp][32 + lane] = s1;
    __syncthreads();
    if (tid < 42) {
      double s = 0.0;
#pragma unroll
      for (int wq = 0; wq < NT / 32; ++wq) s += (double)red[wq][tid];
      if (tid < 36) {
        const int r = tid / 6, c = tid % 6;
        atomicAdd(&H[(size_t)(6 * pa + r) * d.n + 6 * pb + c], -s);
        if (!diag) atomicAdd(&H[(size_t)(6 * pb + c) * d.n + 6 * pa + r], -s);
      } else {
        atomicAdd(&bvec[6 * pa + (tid - 36)], -s);
      }
    }
    __syncthreads();
  };
  for (int u = u0; u < u1; ++u) {
    const int p = u / nchunk;
    const int px0 = (u - p * nchunk) * kChunk;
    const int px1 = min(d.hw, px0 + kChunk);
    if (p != cur) {
      if (cur >= 0) flush();
      cur = p;
      // slot k with pair_ptr[k] <= p < pair_ptr[k+1]
      int k;
      if (M <= 32) {
        const int v = lane < M ? ws.pair_ptr[lane] : 0x7fffffff;
        k = __popc(__ballot_sync(0xffffffffu, v <= p)) - 1;
      } else {
        int lo = 0, hi = M;
        while (hi - lo > 1) {
          const int mid = (lo + hi) >> 1;
          if (ws.pair_ptr[mid] <= p) lo = mid; else hi = mid;
        }
        k = lo;
      }
      const int e0 = ws.entry_ptr[k];
      const int ne = ws.entry_ptr[k + 1] - e0;
      int q = p - ws.pair_ptr[k];
      int a = 0;
      while (q >= ne - a) { q -= ne - a; ++a; }      // row a of the upper triangle
      const int b = a + q;
      const int ca = ws.entry_code[e0 + a];
      const int cb = ws.entry_code[e0 + b];
      Ea = (ca >= 0) ? ws.Eij + (size_t)ca * 6 * d.hw : ws.Ei + (size_t)k * 6 * d.hw;
      Eb = (cb >= 0) ? ws.Eij + (size_t)cb * 6 * d.hw : ws.Ei + (size_t)k * 6 * d.hw;
      pa = (ca >= 0) ? ws.edge_j[ca] - d.t0 : -ca - 1;
      pb = (cb >= 0) ? ws.edge_j[cb] - d.t0 : -cb - 1;
      Qk = ws.Q + (size_t)k * d.hw;
      wk = ws.w + (size_t)k * d.hw;
      diag = a == b;
#pragma unroll
      for (int i = 0; i < 64; ++i) acc[i] = 0.f;
    }
    // predicated, branch-free body: all 4 x 14 loads of the chunk are in flight together
    float qv[kChunk / NT], wv[kChunk / NT], ea[kChunk / NT][6], eb[kChunk / NT][6];
#pragma unroll
    for (int v = 0; v < kChunk / NT; ++v) {
      const int px = px0 + tid + v * NT;
      const bool ok = px < px1;
      qv[v] = ok ? Qk[px] : 0.f;
      wv[v] = (ok && diag) ? wk[px] : 0.f;
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        ea[v][r] = ok ? Ea[(size_t)r * d.hw + px] : 0.f;
        eb[v][r] = ok ? Eb[(size_t)r * d.hw + px] : 0.f;
      }
    }
#pragma unroll
    for (int v = 0; v < kChunk / NT; ++v) {
#pragma unroll
      for (int r = 0; r < 6; ++r) ea[v][r] *= qv[v];
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = 0; c < 6; ++c) acc[r * 6 + c] += ea[v][r] * eb[v][c];
#pragma unroll
      for (int r = 0; r < 6; ++r) acc[36 + r] += ea[v][r] * wv[v];
    }
  }
  if (cur >= 0) flush();
}

__global__ void __launch_bounds__(256)
ba_system_kernel(const float* poses, const int64_t* __restrict__ ii,
                 const int64_t* __restrict__ jj, BaDims d, BaWs ws, int motion_only) {
  __shared__ SysSmem sm;
  if (ws.counts[4]) return;
  system_items<256>(poses, ii, jj, d, ws, motion_only, blockIdx.x, gridDim.x, sm);
}

// ------------------------------------------------------------------------------------
// Multi-GPU split form over PEER MEMORY (goslam_ba_phase1_peers / goslam_ba_phase2_peers): every rank leaves its partial
// reduced camera system in a buffer its peers have mapped (CUDA IPC over NVLink / NVSwitch); the solve kernels sum
// the partial systems WHILE THEY LOAD the matrix into shared memory — in rank order, so every rank factors bit-identical
// numbers — instead of waiting for an NCCL all-reduce, and the back-substitution writes the inverse-depth rows a rank
// owns straight into every replica instead of an all-gather.  Ordering is by epoch flags in peer memory
// (st.release.sys by a one-warp signal kernel after the producing kernels, ld.acquire.sys spin in the consumer).
// ------------------------------------------------------------------------------------
constexpr int kMaxPeers = 8;
struct SysSrc {
  const double* p[kMaxPeers];        // partial systems in rank order (n == 1: the local, complete system)
  int n;
  const unsigned* flags;             // [n] local flag words, flags[r] >= epoch <=> rank r's partial system is complete
  unsigned epoch;
  int* timeout;
};
struct PeerRows {
  float* p[kMaxPeers];               // every replica of disps (n == 0: local only)
  int n;
};

// Plain loads: the peers' buffers were last written before the flags this kernel acquired in peer_wait (whose asm
// "memory" clobbers + barrier keep these loads behind it), L1 holds nothing of them at kernel start, and plain loads let
// the compiler issue all ranks' (and the unrolled neighbours') loads before the first add — a peer load is ~1 us.
__device__ __forceinline__ double sys_at(const SysSrc& s, size_t i) {
  double x[kMaxPeers];
#pragma unroll
  for (int r = 0; r < kMaxPeers; ++r) x[r] = r < s.n ? __ldcg(s.p[r] + i) : 0.0;
  double v = x[0];
#pragma unroll
  for (int r = 1; r < kMaxPeers; ++r) v += x[r];          // rank order; + 0.0 for absent ranks does not change the sum
  return v;
}

// threads 0..n-1 of the block wait for the n flag words; gives up after ~2 s (a dead peer must not hang the GPU)
__device__ __forceinline__ void peer_wait(const unsigned* flags, int n, unsigned epoch, int* timeout) {
  if (n > 1 && (int)threadIdx.x < n) {
    const long long t0 = clock64();
    unsigned v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + threadIdx.x) : "memory");
      if ((int)(v - epoch) >= 0) break;
      if (clock64() - t0 > (1ll << 32)) { if (timeout) *timeout = 1; break; }
    } while (true);
  }
  __syncthreads();
}

__global__ void ba_peer_wait_kernel(const unsigned* flags, int n, unsigned epoch, int* timeout) {
  peer_wait(flags, n, epoch, timeout);
}

// after the kernels that produced the data (same stream): publish `epoch` in word `slot` of every rank's flag row
__global__ void ba_peer_signal_kernel(PeerRows flag_rows, int slot, unsigned epoch) {
  __threadfence_system();
  if ((int)threadIdx.x < flag_rows.n) {
    unsigned* dst = reinterpret_cast<unsigned*>(flag_rows.p[threadIdx.x]) + slot;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(dst), "r"(epoch) : "memory");
  }
}

// ------------------------------------------------------------------------------------
// Damp + Cholesky (float64) + solve + pose retraction.  One block.
// A lives in shared memory when it fits, else in the global scratch.
// ------------------------------------------------------------------------------------
// finish: write dx / status and retract the poses  (:898-931)
__device__ __forceinline__ void solve_finish(float* poses, const BaDims& d, const BaWs& ws,
                                             const double* x, int fail, float* dx_out,
                                             int* status_out, int tid, int nt) {
  for (int i = tid; i < d.n; i += nt) {
    const float val = fail ? 0.0f : (float)x[i];
    ws.dx[i] = val;
    if (dx_out) dx_out[i] = val;
  }
  if (tid == 0 && status_out) *status_out = fail;
}

// eta shape mismatch (see ba_prep_kernel): zero step, status 2, state untouched
__device__ __forceinline__ void bad_argument_step(const BaDims& d, const BaWs& ws, float* dx_out,
                                                  int* status_out, int tid, int nt) {
  for (int i = tid; i < d.n; i += nt) {
    ws.dx[i] = 0.f;
    if (dx_out) dx_out[i] = 0.f;
  }
  if (tid == 0 && status_out) *status_out = 2;
}

__device__ __forceinline__ void retract_poses(float* poses, const BaDims& d, const BaWs& ws, int tid,
                                              int nt) {
  for (int k = tid; k < d.P; k += nt) {
    float* p = poses + 7 * (size_t)(d.t0 + k);
    float t1[3], q1[4];
    gs_retr(ws.dx + 6 * k, p, p + 3, t1, q1);
    p[0] = t1[0]; p[1] = t1[1]; p[2] = t1[2];
    p[3] = q1[0]; p[4] = q1[1]; p[5] = q1[2]; p[6] = q1[3];
  }
}

// Small systems (6P <= kWarpSolveMaxN): blocked right-looking Cholesky with the natural 6x6
// pose blocks, matrix in shared memory, 128 threads, 3 barriers per block column (a local
// window of 8 keyframes is 7 block columns).  The 6x6 diagonal factor is computed redundantly in
// registers; one rsqrt per column and no divisions.  Blocked forward/backward substitution.
struct SolveSmem {
  double Lblk[16][15];   // strictly-lower part of each factored 6x6 diagonal block (P <= 16)
  double xs[6];
  int failed;
};

#ifdef GOSLAM_BA_PROBE
__device__ long long g_solve_probe[8];
__device__ int g_phase_cycles[2][1024];
#define SOLVE_PROBE(slot) do { if (threadIdx.x == 0) g_solve_probe[slot] = clock64(); } while (0)
#else
#define SOLVE_PROBE(slot) do {} while (0)
#endif

// 128 threads; smd = (n*n + 2n) doubles of shared memory.
//  * The right-hand side rides along as row n of the matrix, so the forward substitution happens
//    inside the factorisation (its panel step) and costs no extra pass.
//  * Every thread factors the current 6x6 diagonal block redundantly in registers (21 broadcast
//    loads, one rsqrt per column): no barrier and no shared-memory hop between the block factor
//    and the panel solve.  2 barriers per block column.
//  * Backward substitution is right-looking: solve a block, push it into the rows above.
__device__ __forceinline__ void solve_small(float* poses, const BaDims& d, const BaWs& ws,
                                            const SysSrc& sys_in, float lm, float ep, float* dx_out,
                                            int* status_out, double* smd, SolveSmem& ss) {
  double* xs = ss.xs;
  int& failed = ss.failed;
  const int n = d.n, P = d.P, tid = threadIdx.x, lane = tid & 31;
  double* __restrict__ A = smd;                       // rows 0..n-1: lower triangle; row n: rhs
  double* __restrict__ invd = smd + (size_t)(n + 1) * n;   // 1/l_jj
  SOLVE_PROBE(0);
  // the pose this thread will retract, fetched now so that its latency hides under the factorisation
  float pose_old[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f};
  if (tid < P) {
#pragma unroll
    for (int c = 0; c < 7; ++c) pose_old[c] = poses[7 * (size_t)(d.t0 + tid) + c];
  }
  // ---- load (lower triangle + rhs row), damping on the diagonal.  All of a thread's loads are
  // issued before the first store: one L2 round trip for a local window (n = 42 -> 15 loads) ----
  {
    const int tot = (n + 1) * n;
    for (int base = 0; base < tot; base += 128 * 16) {
      double v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int idx = base + tid + 128 * u;
        const int r = idx / n, c = idx - r * n;
        v[u] = (idx < tot && (c <= r || r == n)) ? sys_at(sys_in, idx) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int idx = base + tid + 128 * u;
        const int r = idx / n, c = idx - r * n;
        if (idx < tot && (c <= r || r == n)) {
          double val = v[u];
          if (r == c) val += (double)ep + (double)lm * val;
          A[idx] = val;
        }
      }
    }
  }
  if (tid == 0) failed = 0;
  __syncthreads();
  SOLVE_PROBE(1);

  bool bad = false;
  for (int jb = 0; jb < P; ++jb) {
    const int j0 = 6 * jb;
    // (a) 6x6 diagonal block, redundantly per thread
    double l[6][6];
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c <= r; ++c) l[r][c] = A[(j0 + r) * n + j0 + c];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      double dkk = l[k][k];
#pragma unroll
      for (int m = 0; m < k; ++m) dkk -= l[k][m] * l[k][m];
      bad = bad || !(dkk > 0.0);
      const double inv = rsqrt(dkk);
      l[k][k] = inv;
#pragma unroll
      for (int r = k + 1; r < 6; ++r) {
        double v = l[r][k];
#pragma unroll
        for (int m = 0; m < k; ++m) v -= l[r][m] * l[k][m];
        l[r][k] = v * inv;
      }
    }
    if (tid < 6) {                                    // keep L of the block for the back-substitution
      invd[j0 + tid] = l[0][0] * (tid == 0) + l[1][1] * (tid == 1) + l[2][2] * (tid == 2) +
                       l[3][3] * (tid == 3) + l[4][4] * (tid == 4) + l[5][5] * (tid == 5);
    } else if (tid == 32) {
      // (not into A: slower threads may still be reading the unfactored block)
#pragma unroll
      for (int r = 1; r < 6; ++r)
#pragma unroll
        for (int c = 0; c < r; ++c) ss.Lblk[jb][r * (r - 1) / 2 + c] = l[r][c];
    }
    // (b) panel: rows below the block (and the rhs row), x L_d^T = a_row
    for (int i = j0 + 6 + tid; i <= n; i += 128) {
      double x[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) x[k] = A[i * n + j0 + k];
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        double v = x[k];
#pragma unroll
        for (int m = 0; m < k; ++m) v -= x[m] * l[k][m];
        x[k] = v * l[k][k];
      }
#pragma unroll
      for (int k = 0; k < 6; ++k) A[i * n + j0 + k] = x[k];
    }
    __syncthreads();
    // (c) rank-6 update of the trailing lower triangle and of the rhs row.
    // 4 threads per row (columns c = t, t+4, ...), 32 rows per pass.
    {
      const int t4 = tid & 3;
      for (int i = j0 + 6 + (tid >> 2); i <= n; i += 32) {
        double ri[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) ri[k] = A[i * n + j0 + k];
        const int cend = i < n ? i : n - 1;
        for (int c = j0 + 6 + t4; c <= cend; c += 4) {
          double acc = A[i * n + c];
#pragma unroll
          for (int k = 0; k < 6; ++k) acc -= ri[k] * A[c * n + j0 + k];
          A[i * n + c] = acc;
        }
      }
    }
    __syncthreads();
  }
  if (bad && tid == 0) failed = 1;
  __syncthreads();
  SOLVE_PROBE(2);

  double* __restrict__ y = A + (size_t)n * n;        // row n = L^-1 b
  int fail = failed;
  if (!fail) {
    // backward: L^T x = z, right-looking
    for (int jb = P - 1; jb >= 0; --jb) {
      const int j0 = 6 * jb;
      if (tid == 0) {
        double lt[6][6], x[6], iv[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) { x[k] = y[j0 + k]; iv[k] = invd[j0 + k]; }
#pragma unroll
        for (int r = 1; r < 6; ++r)
#pragma unroll
          for (int c = 0; c < r; ++c) lt[r][c] = ss.Lblk[jb][r * (r - 1) / 2 + c];
#pragma unroll
        for (int k = 5; k >= 0; --k) {
          double v = x[k];
#pragma unroll
          for (int mm = k + 1; mm < 6; ++mm) v -= lt[mm][k] * x[mm];
          x[k] = v * iv[k];
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) { y[j0 + k] = x[k]; xs[k] = x[k]; }
      }
      __syncthreads();
      for (int i = tid; i < j0; i += 128) {
        double v = y[i];
#pragma unroll
        for (int k = 0; k < 6; ++k) v -= A[(j0 + k) * n + i] * xs[k];
        y[i] = v;
      }
      __syncthreads();
    }
    if (tid < 32) {
      int nf = 0;
      for (int i = lane; i < n; i += 32) nf |= !isfinite(y[i]);
      if (__any_sync(0xffffffffu, nf) && lane == 0) failed = 1;
    }
    __syncthreads();
    fail = failed;
  }
  SOLVE_PROBE(3);
  solve_finish(poses, d, ws, y, fail, dx_out, status_out, tid, 128);
  if (tid < P) {                                       // P <= 16: one pose per thread, dx straight from smem
    float xi[6], t1[3], q1[4];
#pragma unroll
    for (int c = 0; c < 6; ++c) xi[c] = fail ? 0.0f : (float)y[6 * tid + c];
    gs_retr(xi, pose_old, pose_old + 3, t1, q1);
    float* p = poses + 7 * (size_t)(d.t0 + tid);
    p[0] = t1[0]; p[1] = t1[1]; p[2] = t1[2];
    p[3] = q1[0]; p[4] = q1[1]; p[5] = q1[2]; p[6] = q1[3];
  }
  SOLVE_PROBE(4);
}

__global__ void __launch_bounds__(128)
ba_solve_warp_kernel(float* poses, BaDims d, BaWs ws, const SysSrc sys_in, float lm, float ep,
                     float* dx_out, int* status_out) {
  extern __shared__ double smd[];
  __shared__ SolveSmem ss;
  if (ws.counts[4]) { bad_argument_step(d, ws, dx_out, status_out, threadIdx.x, blockDim.x); return; }
  peer_wait(sys_in.flags, sys_in.n, sys_in.epoch, sys_in.timeout);
  solve_small(poses, d, ws, sys_in, lm, ep, dx_out, status_out, smd, ss);
}

// General case: one block; A in shared memory when it fits, else in the global scratch.
__global__ void __launch_bounds__(1024)
ba_solve_kernel(float* __restrict__ poses, BaDims d, BaWs ws, const SysSrc sys_in,
                float lm, float ep, int use_smem, float* __restrict__ dx_out,
                int* __restrict__ status_out) {
  extern __shared__ double smd[];
  __shared__ int fail;
  const int n = d.n, tid = threadIdx.x, nt = blockDim.x;
  if (ws.counts[4]) { bad_argument_step(d, ws, dx_out, status_out, tid, nt); return; }
  peer_wait(sys_in.flags, sys_in.n, sys_in.epoch, sys_in.timeout);
  double* A = use_smem ? smd : ws.chol;
  double* b = use_smem ? smd + (size_t)n * n : ws.rhs;
  if (tid == 0) fail = 0;
  for (size_t idx = tid; idx < (size_t)n * n; idx += nt) {
    const int r = (int)(idx / n), c = (int)(idx % n);
    double val = sys_at(sys_in, idx);
    if (r == c) val += (double)ep + (double)lm * val;
    A[idx] = val;
  }
  for (int i = tid; i < n; i += nt) b[i] = sys_at(sys_in, (size_t)n * n + i);
  __syncthreads();

  // right-looking Cholesky on the lower triangle; the diagonal keeps 1/l_jj
  for (int j = 0; j < n; ++j) {
    const double ajj = A[(size_t)j * n + j];
    if (!(ajj > 0.0)) { if (tid == 0) fail = 1; }
    __syncthreads();
    if (fail) break;
    const double inv = rsqrt(ajj);
    for (int i = j + 1 + tid; i < n; i += nt) A[(size_t)i * n + j] *= inv;
    if (tid == 0) A[(size_t)j * n + j] = inv;
    __syncthreads();
    const int m = n - j - 1;
    const int tot = m * m;                       // n <= 6*4096 => fits in int
    for (int idx = tid; idx < tot; idx += nt) {
      const int q = idx / m;
      const int i = j + 1 + q, c = j + 1 + (idx - q * m);
      if (c <= i) A[(size_t)i * n + c] -= A[(size_t)i * n + j] * A[(size_t)c * n + j];
    }
    __syncthreads();
  }

  if (!fail) {
    for (int j = 0; j < n; ++j) {
      const double zj = b[j] * A[(size_t)j * n + j];
      __syncthreads();
      if (tid == 0) b[j] = zj;
      for (int i = j + 1 + tid; i < n; i += nt) b[i] -= A[(size_t)i * n + j] * zj;
      __syncthreads();
    }
    for (int j = n - 1; j >= 0; --j) {
      const double xj = b[j] * A[(size_t)j * n + j];
      __syncthreads();
      if (tid == 0) b[j] = xj;
      for (int i = tid; i < j; i += nt) b[i] -= A[(size_t)j * n + i] * xj;
      __syncthreads();
    }
    int bad = 0;
    for (int i = tid; i < n; i += nt) bad |= !isfinite(b[i]);
    if (bad) fail = 1;
    __syncthreads();
  }
  solve_finish(poses, d, ws, b, fail, dx_out, status_out, tid, nt);
  __syncthreads();
  retract_poses(poses, d, ws, tid, nt);
}

// ------------------------------------------------------------------------------------
// Global-BA-sized systems (96 < 6P, up to ~100 poses): ONE THREAD-BLOCK CLUSTER of kCl CTAs holds
// the lower triangle of the reduced camera matrix in DISTRIBUTED SHARED MEMORY (6x6 pose blocks,
// block row r lives in CTA r % kCl) and runs the same right-looking 6x6-blocked Cholesky as
// solve_small, with hardware cluster barriers between the phases of a block column:
//   (A) the 6x6 diagonal block is fetched from its owner (36 DSMEM loads) and factored redundantly
//       in registers by the threads that need it; (B) every CTA solves the panel blocks of ITS rows
//       (and its replica of the right-hand-side row: forward substitution rides along);
//   --- cluster barrier --- (C) the block column is gathered from its owners into a local buffer
//   (DSMEM loads, <= 9 per thread) and (D) the trailing update of the CTA's own rows runs out of local
//   shared memory; --- cluster barrier ---.
// Backward substitution: right-looking over block rows, each owner folding x_jb into a LOCAL vector of
// partial sums that the next owner collects through DSMEM; one cluster barrier per block row.
// P = 63 (config 4): 378 unknowns, 80 KB of matrix per CTA.  Replaces a single-block factorisation out
// of global scratch that needed 5.2 ms per solve (tools/time_ba_large.py) — the reference does this
// step on the host with Eigen SimplicialLLT (src/lib/droid_kernels.cu:1192-1213).
// ------------------------------------------------------------------------------------
constexpr int kCl = 8;        // portable cluster size
constexpr int kClT = 512;     // threads per CTA

__host__ __device__ inline int cl_row_off(int q, int l) {      // doubles before local block row l of CTA q
  return 36 * (l * (q + 1) + kCl * (l * (l - 1) / 2));
}
inline size_t cl_rows_doubles(int P) {                         // largest per-CTA matrix slice
  size_t mx = 0;
  for (int q = 0; q < kCl; ++q) {
    const int nl = (P - q + kCl - 1) / kCl;
    if (nl > 0) mx = std::max(mx, (size_t)cl_row_off(q, nl));
  }
  return mx;
}
// rows | rhs[n] | ps[n] | panel[P][36] | dloc[36] | xs[16] | inbox[kCl][6]
inline size_t cl_smem_bytes(int P) {
  return (cl_rows_doubles(P) + 2 * (size_t)(6 * P) + (size_t)P * 36 + 36 + 16 + kCl * 6) * sizeof(double);
}

// Everything that crosses CTAs is PUSHED (remote stores, fire and forget) ahead of the cluster barrier that
// publishes it, so no phase starts with a round trip through distributed shared memory:
//   panel blocks  -> every CTA's `panel`   (by their owners, after the panel solve)
//   next diagonal -> every CTA's `dloc`    (by its owner, as soon as its own row is updated)
//   backward pass -> partial sums of the next 8 block rows go to their owners' `inbox`
__global__ void __launch_bounds__(kClT)
ba_solve_cluster_kernel(float* poses, BaDims d, BaWs ws, const SysSrc sys_in, float lm,
                        float ep, int rows_doubles, float* dx_out, int* status_out) {
  namespace cg = cooperative_groups;
  extern __shared__ double smd[];
  __shared__ int failed;
  cg::cluster_group cluster = cg::this_cluster();
  const int q = (int)cluster.block_rank();
  const int P = d.P, n = d.n, tid = threadIdx.x;
  if (ws.counts[4]) {                                  // uniform over the cluster
    if (q == 0) bad_argument_step(d, ws, dx_out, status_out, tid, kClT);
    return;
  }
  double* rows = smd;                                  // own block rows, row l = blocks 0..r (r = q + l*kCl)
  double* rhs = smd + rows_doubles;                    // [n]  replica of the right-hand side -> y = L^-1 b
  double* ps = rhs + n;                                // [n]  backward substitution: local partial sums
  double* panel = ps + n;                              // [P][36] block column of the current step (pushed in)
  double* dloc = panel + (size_t)P * 36;               // [36] diagonal block of the current step (pushed in)
  double* xs = dloc + 36;                              // [6] + [6]
  double* inbox = xs + 16;                             // [kCl][6]: partial sums from CTA s for my NEXT own block row
  const int nl = (P - q + kCl - 1) / kCl;              // own block rows (may be <= 0 for tiny P)
  double* peer_panel[kCl];
  double* peer_dloc[kCl];
#pragma unroll
  for (int oq = 0; oq < kCl; ++oq) {
    peer_panel[oq] = cluster.map_shared_rank(panel, oq);
    peer_dloc[oq] = cluster.map_shared_rank(dloc, oq);
  }

  // every CTA reads partial systems itself: each waits for the ranks' flags (no-op for a local system)
  peer_wait(sys_in.flags, sys_in.n, sys_in.epoch, sys_in.timeout);
  // ---- load own rows (lower blocks incl. the diagonal one), damping on the diagonal
  for (int l = 0; l < nl; ++l) {
    const int r = q + l * kCl;
    double* dst = rows + cl_row_off(q, l);
    const int width = 6 * (r + 1);
#pragma unroll 4
    for (int idx = tid; idx < 6 * width; idx += kClT) {
      const int a = idx / width, col = idx - a * width;
      double val = sys_at(sys_in, (size_t)(6 * r + a) * n + col);
      if (col == 6 * r + a) val += (double)ep + (double)lm * val;
      dst[(col / 6) * 36 + a * 6 + (col % 6)] = val;
    }
  }
  for (int i = tid; i < n; i += kClT) { rhs[i] = sys_at(sys_in, (size_t)n * n + i); ps[i] = 0.0; }
  for (int i = tid; i < kCl * 6; i += kClT) inbox[i] = 0.0;
  if (tid == 0) failed = 0;
  // every CTA of the cluster must be running before anybody stores into its shared memory (compute-sanitizer:
  // "block that might not have entered yet"); also orders the loads above with the factor below
  cluster.sync();
  // 6x6 Cholesky of a diagonal block held in shared memory (lower triangle); leaves L^-1 (lower triangular) in
  // its place.  With the explicit inverse, the panel solve X = A L^-T, the forward substitution of the right-hand
  // side and the backward solve x = L^-T v are 6 INDEPENDENT dot products instead of a 21-deep chain of dependent
  // fp64 operations (a dependent DFMA costs ~50 cycles here; probes: profiles/r02_cluster_solve.md).  The blocks
  // are damped 6x6 pose blocks, far from singular; the factorisation itself stays a Cholesky.
  // One thread; returns false when a pivot is not positive.
  auto factor_block = [](double* blk) -> bool {
    double l[6][6];
    bool ok = true;
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c <= r; ++c) l[r][c] = blk[r * 6 + c];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      double dkk = l[k][k];
#pragma unroll
      for (int m = 0; m < k; ++m) dkk -= l[k][m] * l[k][m];
      ok = ok && (dkk > 0.0);
      const double inv = rsqrt(dkk);
      l[k][k] = inv;
#pragma unroll
      for (int r = k + 1; r < 6; ++r) {
        double v = l[r][k];
#pragma unroll
        for (int m = 0; m < k; ++m) v -= l[r][m] * l[k][m];
        l[r][k] = v * inv;
      }
    }
    // in-place inverse of the lower-triangular factor (l[k][k] already holds 1/l_kk), column by column
    double li[6][6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      li[k][k] = l[k][k];
#pragma unroll
      for (int r = k + 1; r < 6; ++r) {
        double v = 0.0;
#pragma unroll
        for (int m = k; m < r; ++m) v -= l[r][m] * li[m][k];
        li[r][k] = v * l[r][r];
      }
    }
#pragma unroll
    for (int r = 0; r < 6; ++r)
#pragma unroll
      for (int c = 0; c <= r; ++c) blk[r * 6 + c] = li[r][c];
    return ok;
  };
  constexpr int kFG = 64;                              // "factor group": threads 0..63 of the next row's owner
  if (q == 0) {                                        // first diagonal block: factor, then to everyone
    if (tid == 0 && !factor_block(rows)) failed = 1;
    __syncthreads();
    if (tid < 36) {
      const double v = rows[tid];
#pragma unroll
      for (int oq = 0; oq < kCl; ++oq) peer_dloc[oq][tid] = v;
    }
  }
  cluster.sync();

#ifdef GOSLAM_BA_PROBE
  long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long pt0 = clock64();
#define CL_PROBE(i) do { const long long t__ = clock64(); pc[i] += t__ - pt0; pt0 = t__; } while (0)
#else
#define CL_PROBE(i) do {} while (0)
#endif
  for (int jb = 0; jb < P; ++jb) {
    // first own block row below jb
    const int l0 = jb < q ? 0 : (jb - q) / kCl + 1;
    const int npan = nl > l0 ? nl - l0 : 0;
    // (A) panel solve of own rows with L_d^-1 of the diagonal block, which its owner pushed into dloc
    if (tid < 6 * npan || tid == 0) {
      double l[6][6];
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = 0; c <= r; ++c) l[r][c] = dloc[r * 6 + c];
      if (tid < 6 * npan) {                           // one scalar row of one own block per thread
        const int lr = l0 + tid / 6, a = tid % 6;
        double* blk = rows + cl_row_off(q, lr) + jb * 36 + a * 6;
        double x[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) x[k] = blk[k];
#pragma unroll
        for (int k = 0; k < 6; ++k) {                 // X = A L^-T: row a of the block times column k of L^-T
          double v = x[0] * l[k][0];
#pragma unroll
          for (int m = 1; m <= k; ++m) v += x[m] * l[k][m];
          blk[k] = v;
        }
      }
      if (tid == 0) {                                 // right-hand-side row (replicated in every CTA)
        double x[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) x[k] = rhs[6 * jb + k];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          double v = x[0] * l[k][0];
#pragma unroll
          for (int m = 1; m <= k; ++m) v += x[m] * l[k][m];
          rhs[6 * jb + k] = v; xs[k] = v;
        }
      }
    }
    __syncthreads();
    // push own panel blocks into every CTA's panel buffer
    for (int idx = tid; idx < npan * 36 * kCl; idx += kClT) {
      const int oq = idx % kCl, e = (idx / kCl) % 36, m = idx / (kCl * 36);
      const int r = q + (l0 + m) * kCl;
      peer_panel[oq][(size_t)r * 36 + e] = rows[cl_row_off(q, l0 + m) + jb * 36 + e];
    }
    CL_PROBE(0);
    cluster.sync();                                   // the whole block column is in every CTA
    CL_PROBE(1);
    // (D0) In the CTA that owns block row jb+1, threads 0..63 update that row's diagonal block, factor it and
    // push L_d to every CTA WHILE the other threads (and the other CTAs) do their trailing updates: the
    // 6 sequential pivots (~1.5 k cycles of dependent fp64) are off the critical path.
    const bool next_owner = (q == (jb + 1) % kCl) && (jb + 1 < P);
    const bool in_fg = next_owner && tid < kFG;
    if (in_fg) {
      double* rowp = rows + cl_row_off(q, (jb + 1) / kCl);
      double* dblk = rowp + (jb + 1) * 36;
      if (tid < 36) {
        const int a = tid / 6, b = tid % 6;
        const double* Li = rowp + jb * 36;
        double v = dblk[tid];
#pragma unroll
        for (int k = 0; k < 6; ++k) v -= Li[a * 6 + k] * Li[b * 6 + k];
        dblk[tid] = v;
      }
      asm volatile("bar.sync 1, 64;" ::: "memory");
      if (tid == 0 && !factor_block(dblk)) failed = 1;
      asm volatile("bar.sync 1, 64;" ::: "memory");
      if (tid < 36) {
        const double v = dblk[tid];
#pragma unroll
        for (int oq = 0; oq < kCl; ++oq) peer_dloc[oq][tid] = v;
      }
    } else {
      // (D) trailing update of own rows: A[i,c] -= L[i,jb] L[c,jb]^T, jb < c <= i; items (row, c, scalar row a)
      // flattened over the CTA's rows: row m (block row r = rb + kCl*m) has 6 * (base + kCl*m) items
      const int ut = next_owner ? tid - kFG : tid, un = next_owner ? kClT - kFG : kClT;
      if (npan > 0) {
        const int base = q + l0 * kCl - jb;           // blocks of the first own row below jb (1..kCl)
        const int total = 6 * (base * npan + (kCl / 2) * npan * (npan - 1));
        // the next owner's first row is jb+1 itself (one block: the diagonal one, done by the factor group)
        for (int it = ut + (next_owner ? 6 : 0); it < total; it += un) {
          int m = 0, t = it, cnt = 6 * base;
          while (t >= cnt) { t -= cnt; ++m; cnt += 6 * kCl; }
          const int c = jb + 1 + t / 6, a = t % 6;
          double* rowp = rows + cl_row_off(q, l0 + m);
          const double* Li = rowp + jb * 36 + a * 6;
          const double* Lc = panel + (size_t)c * 36;
          double li[6], acc[6];
#pragma unroll
          for (int k = 0; k < 6; ++k) li[k] = Li[k];
          double* out = rowp + c * 36 + a * 6;
#pragma unroll
          for (int b = 0; b < 6; ++b) {
            double v = out[b];
#pragma unroll
            for (int k = 0; k < 6; ++k) v -= li[k] * Lc[b * 6 + k];
            acc[b] = v;
          }
#pragma unroll
          for (int b = 0; b < 6; ++b) out[b] = acc[b];
        }
      }
      // right-hand-side row: b[c] -= y_jb L[c,jb]^T
      for (int it = ut; it < (P - 1 - jb) * 6; it += un) {
        const int c = jb + 1 + it / 6, b = it % 6;
        const double* Lc = panel + (size_t)c * 36 + b * 6;
        double v = rhs[6 * c + b];
#pragma unroll
        for (int k = 0; k < 6; ++k) v -= xs[k] * Lc[k];
        rhs[6 * c + b] = v;
      }
    }
    CL_PROBE(2);
    cluster.sync();                                   // next L_d is in every dloc; panel may be overwritten
    CL_PROBE(3);
  }

  // ---- backward substitution L^T x = y.  Right-looking over block rows: the owner of row jb solves x_jb,
  // folds it into its local partial sums ps[c] += L[jb,c]^T x_jb (c < jb) and pushes the entries of the next
  // kCl block rows — final, because its next own row is jb - kCl — into their owners' inboxes.  Runs even
  // after a failed pivot (NaNs are harmless here; the result is discarded): every CTA must take the same path.
  {
    for (int jb = P - 1; jb >= 0; --jb) {
      const int owner = jb % kCl, lo = jb / kCl;
      if (q == owner) {
        const double* Ld = rows + cl_row_off(q, lo) + jb * 36;
        if (tid == 0) {
          double v6[6], x[6];
#pragma unroll
          for (int k = 0; k < 6; ++k) {
            const double s01 = inbox[0 * 6 + k] + inbox[1 * 6 + k], s23 = inbox[2 * 6 + k] + inbox[3 * 6 + k];
            const double s45 = inbox[4 * 6 + k] + inbox[5 * 6 + k], s67 = inbox[6 * 6 + k] + inbox[7 * 6 + k];
            v6[k] = rhs[6 * jb + k] - ((s01 + s23) + (s45 + s67));
          }
          int nf = 0;
#pragma unroll
          for (int k = 0; k < 6; ++k) {               // x = L_d^-T v (Ld holds L_d^-1)
            double v = Ld[k * 6 + k] * v6[k];
#pragma unroll
            for (int m = k + 1; m < 6; ++m) v += Ld[m * 6 + k] * v6[m];
            x[k] = v;
            nf |= !isfinite(v);
          }
#pragma unroll
          for (int k = 0; k < 6; ++k) { xs[k] = x[k]; ws.dx[6 * jb + k] = (float)x[k]; }
          if (nf) failed = 1;
        }
        __syncthreads();
        const double* rowp = rows + cl_row_off(q, lo);
        // the next kCl block rows first (their sums are pushed), then the rest
        const int cpush = jb < kCl ? jb : kCl;          // rows jb-1 .. jb-cpush
        if (tid < cpush * 6) {
          const int c = jb - 1 - tid / 6, k = tid % 6;
          const double* blk = rowp + c * 36;
          double v = ps[6 * c + k];
#pragma unroll
          for (int m = 0; m < 6; ++m) v += blk[m * 6 + k] * xs[m];
          ps[6 * c + k] = v;
          cluster.map_shared_rank(inbox, c % kCl)[q * 6 + k] = v;     // one slot per sender: a CTA has one own row per kCl rows
        }
        for (int it = tid; it < (jb - cpush) * 6; it += kClT) {
          const int c = it / 6, k = it % 6;
          const double* blk = rowp + c * 36;
          double v = ps[6 * c + k];
#pragma unroll
          for (int m = 0; m < 6; ++m) v += blk[m * 6 + k] * xs[m];
          ps[6 * c + k] = v;
        }
      }
      CL_PROBE(5);
      cluster.sync();
      CL_PROBE(6);
    }
  }
#ifdef GOSLAM_BA_PROBE
  if (tid == 0 && (q == 0 || q == 5))
    printf("[cluster solve probe cta %d, P=%d] panel+push %lld | barrier1 %lld | update (factor hidden) %lld | barrier2 %lld | "
           "backward work %lld | backward barrier %lld (cycles)\n", q, P, pc[0], pc[1], pc[2], pc[3], pc[5], pc[6]);
#endif
  // ---- status, dx, retraction (CTA 0); the others stay until their flags have been read
  if (q == 0) {
    __shared__ int any_fail;
    if (tid == 0) {
      int f = 0;
      for (int oq = 0; oq < kCl; ++oq) f |= *cluster.map_shared_rank(&failed, oq);
      any_fail = f;
    }
    __syncthreads();
    const int fail = any_fail;
    for (int i = tid; i < n; i += kClT) {
      const float val = fail ? 0.0f : ws.dx[i];
      ws.dx[i] = val;
      if (dx_out) dx_out[i] = val;
    }
    if (tid == 0 && status_out) *status_out = fail;
    __syncthreads();
    retract_poses(poses, d, ws, tid, kClT);
  }
  cluster.sync();
}

// ------------------------------------------------------------------------------------
// Depth back-substitution + retraction: dz = Q (w - sum_a E_a^T dx[pose_a]), disps += dz.
// (EvT6x1 + accum + disp_retr, :1095-1115,:1417,:933-946)
// ------------------------------------------------------------------------------------
__device__ __forceinline__ void backsub_tile(float* disps, const BaDims& d, const BaWs& ws,
                                             int owner_lo, int owner_hi, float* dz_out, int k,
                                             int wt, const PeerRows* peers = nullptr) {
  const int f = ws.kx[k];
  if (f < owner_lo || f >= owner_hi) return;
  const int px = wt * 32 + (threadIdx.x & 31);
  if (px >= d.hw) return;
  float acc = 0.f;
  // own pose entry E_i: pose index f - t0, skipped when <= 0 (reference quirk) or >= P
  {
    const int ix = f - d.t0;
    if (ix > 0 && ix < d.P) {
      float dw = 0.f;
#pragma unroll
      for (int a = 0; a < 6; ++a) dw += ws.Ei[((size_t)k * 6 + a) * d.hw + px] * ws.dx[6 * ix + a];
      acc += dw;
    }
  }
  for (int r = ws.row_ptr[f]; r < ws.row_ptr[f + 1]; ++r) {
    const int e = ws.edge_idx[r];
    const int ix = ws.edge_j[e] - d.t0;
    if (ix <= 0 || ix >= d.P) continue;
    float dw = 0.f;
#pragma unroll
    for (int a = 0; a < 6; ++a) dw += ws.Eij[((size_t)e * 6 + a) * d.hw + px] * ws.dx[6 * ix + a];
    acc += dw;
  }
  const size_t o = (size_t)k * d.hw + px;
  const float dz = ws.Q[o] * (ws.w[o] - acc);
  const float nv = disps[(size_t)f * d.hw + px] + dz;
  disps[(size_t)f * d.hw + px] = nv;
  if (peers)                                     // write-through into every other replica (P2P stores)
    for (int r = 0; r < peers->n; ++r)
      if (peers->p[r] != disps) peers->p[r][(size_t)f * d.hw + px] = nv;
  if (dz_out) dz_out[(size_t)f * d.hw + px] = dz;
}

__global__ void __launch_bounds__(kTP)
ba_backsub_kernel(float* disps, BaDims d, BaWs ws, int owner_lo, int owner_hi, float* dz_out, const PeerRows peers) {
  if ((int)blockIdx.y >= ws.counts[0] || ws.counts[4]) return;
  backsub_tile(disps, d, ws, owner_lo, owner_hi, dz_out, blockIdx.y, blockIdx.x * (kTP / 32) + (threadIdx.x >> 5),
               peers.n > 1 ? &peers : nullptr);
}

// ------------------------------------------------------------------------------------
// Small windows: ALL Gauss-Newton iterations of one call in ONE cooperative kernel.  The phases
// are separated by grid barriers instead of kernel boundaries, and the depth back-substitution
// of iteration i runs fused with the linearisation of iteration i+1 (same pixel, same thread).
// 3 grid barriers per iteration replace 5 launches.
// ------------------------------------------------------------------------------------
#ifdef GOSLAM_BA_PROBE
#define BA_PROBE(slot) do { if (threadIdx.x == 0 && blockIdx.x == 0) probe[slot] = clock64(); } while (0)
#else
#define BA_PROBE(slot) do {} while (0)
#endif

__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned& epoch) {
  __syncthreads();
  ++epoch;
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    const unsigned target = epoch * gridDim.x;
    unsigned v;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
    } while (v < target);
    __threadfence();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kTP)
ba_persistent_kernel(float* poses, float* disps, BaIn in, BaDims d, BaWs ws, int iterations, float lm,
                     float ep, int motion_only, float* dx_out, float* dz_out, int* status_out,
                     unsigned* barrier) {
  extern __shared__ double smd[];
  __shared__ SysSmem sys_sm;
  __shared__ SolveSmem solve_sm;
  unsigned epoch = 0;
#ifdef GOSLAM_BA_PROBE
  __shared__ long long probe[8];
#endif
  const int M = ws.counts[0];
  // linearise / back-substitute unit = (frame slot, 32-pixel warp tile), one per WARP.  Units are dealt
  // warp-major (unit u -> block u % G, warp u / G) so that a partial last round leaves every SM with
  // the same number of busy warps instead of some blocks with four and others with none.
  const int nwt = ws.ntiles * (kTP / 32);
  const int units = M * nwt;
  const int ufirst = (threadIdx.x >> 5) * gridDim.x + blockIdx.x, ustep = (kTP / 32) * gridDim.x;
  const size_t nsys = (size_t)d.n * d.n + d.n;
  if (dz_out) {                      // rows of frames without a depth update stay 0 (first written after 3 barriers)
    const size_t ndz = (size_t)d.num * d.hw;
    for (size_t i = (size_t)blockIdx.x * kTP + threadIdx.x; i < ndz; i += (size_t)gridDim.x * kTP) dz_out[i] = 0.f;
  }
  if (ws.counts[4]) {                 // uniform across the grid: nobody reaches a barrier
    if (blockIdx.x == 0) {
      bad_argument_step(d, ws, dx_out, nullptr, threadIdx.x, kTP);
      if (status_out) for (int it = threadIdx.x; it < iterations; it += kTP) status_out[it] = 2;
    }
    return;
  }
  for (int it = 0; it < iterations; ++it) {
    BA_PROBE(0);
#ifdef GOSLAM_BA_PROBE
    const long long tl0 = clock64();
#endif
    for (int u = ufirst; u < units; u += ustep) {
      const int k = u / nwt, wt = u - k * nwt;
      if (it > 0 && !motion_only) backsub_tile(disps, d, ws, 0, d.num, dz_out, k, wt);
      linearize_tile(in, d, ws, motion_only, k, wt);
    }
#ifdef GOSLAM_BA_PROBE
    if (threadIdx.x == 0 && blockIdx.x < 1024) g_phase_cycles[0][blockIdx.x] = (int)(clock64() - tl0);
#endif
    BA_PROBE(1);
    grid_barrier(barrier, epoch);
    BA_PROBE(2);
#ifdef GOSLAM_BA_PROBE
    const long long ts0 = clock64();
#endif
    system_items<kTP>(poses, in.ii, in.jj, d, ws, motion_only, blockIdx.x, gridDim.x, sys_sm);
#ifdef GOSLAM_BA_PROBE
    if (threadIdx.x == 0 && blockIdx.x < 1024) g_phase_cycles[1][blockIdx.x] = (int)(clock64() - ts0);
#endif
    BA_PROBE(3);
    grid_barrier(barrier, epoch);
    BA_PROBE(4);
    if (blockIdx.x == 0) {
      SysSrc local{};
      local.p[0] = ws.sys; local.n = 1;
      solve_small(poses, d, ws, local, lm, ep, dx_out, status_out ? status_out + it : nullptr, smd,
                  solve_sm);
      __syncthreads();
      for (size_t i = threadIdx.x; i < nsys; i += kTP) ws.sys[i] = 0.0;   // for the next iteration
    }
    BA_PROBE(5);
    grid_barrier(barrier, epoch);
    BA_PROBE(6);
#ifdef GOSLAM_BA_PROBE
    if (threadIdx.x == 0 && blockIdx.x == 0 && it == iterations - 1) {
      for (int ph = 0; ph < 2; ++ph) {
        int mx = 0, arg = 0;
        for (int b = 0; b < (int)gridDim.x && b < 1024; ++b)
          if (g_phase_cycles[ph][b] > mx) { mx = g_phase_cycles[ph][b]; arg = b; }
        printf("[phase %d] slowest block %d: %d cycles; blocks 0/100/200/244/250/270/290/295: %d %d %d %d %d %d %d %d\n", ph, arg,
               mx, g_phase_cycles[ph][0], g_phase_cycles[ph][100], g_phase_cycles[ph][200], g_phase_cycles[ph][244],
               g_phase_cycles[ph][250], g_phase_cycles[ph][270], g_phase_cycles[ph][290], g_phase_cycles[ph][295]);
      }
    }
    if (threadIdx.x == 0 && blockIdx.x == 0)
      printf("[solve probe it=%d] load %lld | factor %lld | backward %lld | finish+retract %lld\n", it,
             g_solve_probe[1] - g_solve_probe[0], g_solve_probe[2] - g_solve_probe[1],
             g_solve_probe[3] - g_solve_probe[2], g_solve_probe[4] - g_solve_probe[3]);
    if (threadIdx.x == 0 && blockIdx.x == 0)
      printf("[ba probe it=%d] linearize %lld | barrier %lld | system %lld | barrier %lld | solve %lld | barrier %lld (cycles)\n",
             it, probe[1] - probe[0], probe[2] - probe[1], probe[3] - probe[2], probe[4] - probe[3],
             probe[5] - probe[4], probe[6] - probe[5]);
#endif
  }
  if (!motion_only)
    for (int u = ufirst; u < units; u += ustep) {
      const int k = u / nwt, wt = u - k * nwt;
      backsub_tile(disps, d, ws, 0, d.num, dz_out, k, wt);
    }
}

bool make_dims(int N, int num, int ht, int wd, int t0, int t1, BaDims* d) {
  if (N < 0 || num <= 0 || num > 4096 || ht <= 0 || wd <= 0) return false;
  d->N = N; d->num = num; d->ht = ht; d->wd = wd; d->hw = ht * wd;
  d->t0 = t0; d->t1 = t1; d->P = t1 - t0 > 0 ? t1 - t0 : 0; d->n = 6 * d->P;
  if (t0 < 0 || t1 > num) return false;
  return true;
}

constexpr int kSmemSolveMaxN = 160;   // (160*160 + 160) * 8 B = 206 KB of the 227 KB
constexpr int kWarpSolveMaxN = 96;    // single-warp solve up to 16 poses
constexpr size_t kClusterSmemMax = 226 * 1024;   // dynamic part of the 227 KB per-CTA opt-in maximum (static: a few bytes)

inline size_t prep_smem_bytes(int num) { return ((size_t)3 * num + 1 + 33) * sizeof(int); }

// Function attributes (opt-in dynamic shared memory) and the occupancy of the cooperative kernel are PER DEVICE.
GsDeviceOnce g_ba_once;
int g_blocks_per_sm[kGsMaxDevices];     // 0: cooperative launch unavailable -> multi-kernel driver

cudaError_t ba_device_init(int dev) {
  const size_t smem_max = ((size_t)kWarpSolveMaxN * kWarpSolveMaxN + 2 * kWarpSolveMaxN) * sizeof(double);
  constexpr cudaFuncAttribute kSmem = cudaFuncAttributeMaxDynamicSharedMemorySize;
  cudaError_t e = cudaFuncSetAttribute(ba_prep_kernel, kSmem, (int)prep_smem_bytes(kPrepMaxFrames));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(ba_solve_kernel, kSmem, (int)(((size_t)kSmemSolveMaxN * kSmemSolveMaxN + kSmemSolveMaxN) * 8));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ba_solve_warp_kernel, kSmem, (int)smem_max);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ba_solve_cluster_kernel, kSmem, (int)kClusterSmemMax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ba_persistent_kernel, kSmem, (int)smem_max);
  if (e != cudaSuccess) return e;
  int occ = 0, coop = 0;
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ba_persistent_kernel, kTP, smem_max);
  constexpr int kWant = 2;    // 2 blocks/SM measured best (profiles/r01: 1 -> 151 us, 2 -> 121 us, 3 -> 124 us)
  g_blocks_per_sm[dev] = (!coop || occ < 1) ? 0 : (occ > kWant ? kWant : occ);
  return cudaSuccess;
}


int launch_phase1(const float* poses, const float* disps, const float* intr,
                  const float* disps_sens, const float* targets, const float* weights,
                  const float* eta, int eta_rows, const int64_t* ii, const int64_t* jj,
                  const BaDims& d, const BaWs& ws, int motion_only, bool prep, cudaStream_t st) {
  const BaIn in{poses, disps, intr, disps_sens, targets, weights, eta, eta_rows, ii, jj};
  if (prep) {
    ba_prep_kernel<<<1, kPrepThreads, prep_smem_bytes(d.num), st>>>(ii, jj, d, ws, 0, motion_only ? 0 : eta_rows);
    GS_CHECK_LAUNCH();
  }
  cudaMemsetAsync(ws.sys, 0, ((size_t)d.n * d.n + d.n) * sizeof(double), st);
  if (d.N > 0) {
    dim3 grid(ws.ntiles, d.num);
    ba_linearize_kernel<<<grid, kTP, 0, st>>>(in, d, ws, motion_only);
    GS_CHECK_LAUNCH();
  } else if (!motion_only) {
    dim3 grid(ws.ntiles, d.num);   // still need Q / w / Ei (= prior only) for every slot
    ba_linearize_kernel<<<grid, kTP, 0, st>>>(in, d, ws, motion_only);
    GS_CHECK_LAUNCH();
  }
  ba_system_kernel<<<148 * 4, 256, 0, st>>>(poses, ii, jj, d, ws, motion_only);
  GS_CHECK_LAUNCH();
  return GOSLAM_OK;
}

int launch_phase2(float* poses, float* disps, const SysSrc& sys_in,
                  const BaDims& d, const BaWs& ws, float lm, float ep, int motion_only,
                  int owner_lo, int owner_hi, float* dx_out, float* dz_out, int* status_out,
                  cudaStream_t st, const PeerRows& peer_rows = PeerRows{}) {
  { const int rc = gs_device_once(g_ba_once, ba_device_init); if (rc != GOSLAM_OK) return rc; }
  if (d.n <= kWarpSolveMaxN) {
    const size_t smem = ((size_t)d.n * d.n + 2 * d.n) * sizeof(double);
    ba_solve_warp_kernel<<<1, 128, smem, st>>>(poses, d, ws, sys_in, lm, ep, dx_out, status_out);
  } else if (cl_smem_bytes(d.P) <= kClusterSmemMax) {
    // one 8-CTA cluster, matrix in distributed shared memory
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kCl);
    cfg.blockDim = dim3(kClT);
    cfg.dynamicSmemBytes = cl_smem_bytes(d.P);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kCl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const int rows_doubles = (int)cl_rows_doubles(d.P);
    const cudaError_t le = cudaLaunchKernelEx(&cfg, ba_solve_cluster_kernel, poses, d, ws, sys_in, lm, ep,
                                              rows_doubles, dx_out, status_out);
    if (le != cudaSuccess) { gs_note_cuda_error(le); return GOSLAM_ELAUNCH; }
  } else {
    const int use_smem = d.n <= kSmemSolveMaxN;
    const size_t smem = use_smem ? ((size_t)d.n * d.n + d.n) * sizeof(double) : 0;
    const int threads = d.n <= kSmemSolveMaxN ? 256 : 1024;
    ba_solve_kernel<<<1, threads, smem, st>>>(poses, d, ws, sys_in, lm, ep, use_smem, dx_out,
                                              status_out);
  }
  GS_CHECK_LAUNCH();
  if (!motion_only) {
    dim3 grid(ws.ntiles, d.num);
    ba_backsub_kernel<<<grid, kTP, 0, st>>>(disps, d, ws, owner_lo, owner_hi, dz_out, peer_rows);
    GS_CHECK_LAUNCH();
  }
  return GOSLAM_OK;
}

}  // namespace

extern "C" {

size_t goslam_ba_workspace_bytes(int N, int num, int ht, int wd, int t0, int t1) {
  BaDims d;
  if (!make_dims(N, num, ht, wd, t0, t1, &d)) return 0;
  return ba_layout(d, nullptr, 0, nullptr) + 256;
}

size_t goslam_ba_system_doubles(int t0, int t1) {
  const size_t n = 6 * (size_t)(t1 > t0 ? t1 - t0 : 0);
  return n * n + n;
}

int goslam_ba(float* poses, float* disps, const float* intrinsics, const float* disps_sens,
              const float* targets, const float* weights, const float* eta, int eta_rows,
              const int64_t* ii, const int64_t* jj, int N, int num, int ht, int wd, int t0,
              int t1, int iterations, float lm, float ep, int motion_only, float* dx_out,
              float* dz_out, int* status_out, void* workspace, size_t workspace_bytes,
              void* stream) {
  BaDims d;
  if (!make_dims(N, num, ht, wd, t0, t1, &d)) return GOSLAM_EINVAL;
  if (!motion_only && (eta == nullptr || eta_rows == 0)) return GOSLAM_EINVAL;
  if (d.P == 0 || iterations <= 0) return GOSLAM_OK;
  BaWs ws;
  const size_t need = ba_layout(d, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  if (d.n <= kWarpSolveMaxN) {
    { const int rc = gs_device_once(g_ba_once, ba_device_init); if (rc != GOSLAM_OK) return rc; }
    int dev = 0;
    cudaGetDevice(&dev);
    const int blocks_per_sm = g_blocks_per_sm[dev], sms = gs_sm_count();
    const size_t smem = ((size_t)d.n * d.n + 2 * d.n) * sizeof(double);
    if (blocks_per_sm > 0) {
      // two launches per call: the table kernel (which also zeroes the reduced system and the barrier
      // counter) and the cooperative kernel (which zeroes dz_out itself)
      ba_prep_kernel<<<1, kPrepThreads, prep_smem_bytes(d.num), st>>>(ii, jj, d, ws, 1, motion_only ? 0 : eta_rows);
      GS_CHECK_LAUNCH();
      unsigned* barrier = reinterpret_cast<unsigned*>(ws.counts + 3);
      BaIn in{poses, disps, intrinsics, disps_sens, targets, weights, eta, eta_rows, ii, jj};
      BaDims dd = d;
      BaWs wsv = ws;
      void* args[] = {&poses, &disps, &in, &dd, &wsv, &iterations, &lm, &ep, &motion_only,
                      &dx_out, &dz_out, &status_out, &barrier};
      const cudaError_t le = cudaLaunchCooperativeKernel((const void*)ba_persistent_kernel,
                                                         dim3(sms * blocks_per_sm), dim3(kTP), args, smem, st);
      if (le != cudaSuccess) { gs_note_cuda_error(le); return GOSLAM_ELAUNCH; }
      return GOSLAM_OK;
    }
  }
  if (dz_out) cudaMemsetAsync(dz_out, 0, (size_t)num * d.hw * sizeof(float), st);
  for (int it = 0; it < iterations; ++it) {
    int rc = launch_phase1(poses, disps, intrinsics, disps_sens, targets, weights, eta, eta_rows,
                           ii, jj, d, ws, motion_only, it == 0, st);
    if (rc) return rc;
    SysSrc local{};
    local.p[0] = ws.sys; local.n = 1;
    rc = launch_phase2(poses, disps, local, d, ws, lm, ep, motion_only, 0, num, dx_out,
                       dz_out, status_out ? status_out + it : nullptr, st);
    if (rc) return rc;
  }
  return GOSLAM_OK;
}

int goslam_ba_phase1(const float* poses, const float* disps, const float* intrinsics,
                     const float* disps_sens, const float* targets, const float* weights,
                     const float* eta, int eta_rows, const int64_t* ii, const int64_t* jj, int N,
                     int num, int ht, int wd, int t0, int t1, int motion_only, double* system,
                     void* workspace, size_t workspace_bytes, void* stream) {
  BaDims d;
  if (!make_dims(N, num, ht, wd, t0, t1, &d)) return GOSLAM_EINVAL;
  if (d.P == 0) return GOSLAM_OK;
  BaWs ws;
  const size_t need = ba_layout(d, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_phase1(poses, disps, intrinsics, disps_sens, targets, weights, eta, eta_rows, ii,
                         jj, d, ws, motion_only, true, st);
  if (rc) return rc;
  if (system != ws.sys)
    cudaMemcpyAsync(system, ws.sys, ((size_t)d.n * d.n + d.n) * sizeof(double),
                    cudaMemcpyDeviceToDevice, st);
  return GOSLAM_OK;
}

int goslam_ba_phase2(float* poses, float* disps, const double* system, int N, int num, int ht,
                     int wd, int t0, int t1, float lm, float ep, int motion_only, int owner_lo,
                     int owner_hi, float* dx_out, float* dz_out, int* status_out, void* workspace,
                     size_t workspace_bytes, void* stream) {
  BaDims d;
  if (!make_dims(N, num, ht, wd, t0, t1, &d)) return GOSLAM_EINVAL;
  if (d.P == 0) return GOSLAM_OK;
  BaWs ws;
  const size_t need = ba_layout(d, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  SysSrc local{};
  local.p[0] = system; local.n = 1;
  return launch_phase2(poses, disps, local, d, ws, lm, ep, motion_only, owner_lo, owner_hi, dx_out,
                       dz_out, status_out, (cudaStream_t)stream);
}

static bool peers_ok(const goslam_ba_peers* p) {
  if (!p || p->world < 1 || p->world > kMaxPeers || p->rank < 0 || p->rank >= p->world || p->epoch == 0) return false;
  for (int r = 0; r < p->world; ++r)
    if (!p->system[r] || !p->flags[r] || !p->disps[r]) return false;
  return true;
}

int goslam_ba_phase1_peers(const float* poses, const float* intrinsics, const float* disps_sens, const float* targets,
                           const float* weights, const float* eta, int eta_rows, const int64_t* ii, const int64_t* jj,
                           int N, int num, int ht, int wd, int t0, int t1, int motion_only,
                           const goslam_ba_peers* peers, void* workspace, size_t workspace_bytes, void* stream) {
  BaDims d;
  if (!make_dims(N, num, ht, wd, t0, t1, &d) || !peers_ok(peers)) return GOSLAM_EINVAL;
  if (d.P == 0) return GOSLAM_OK;
  BaWs ws;
  const size_t need = ba_layout(d, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int W = peers->world, me = peers->rank;
  // (1) every rank has written the inverse-depth rows of the previous iteration into my replica, and has finished
  //     reading my previous partial system (it signals slot [W + r] after its solve + back-substitution)
  if (W > 1) {
    ba_peer_wait_kernel<<<1, 32, 0, st>>>(peers->flags[me] + W, W, peers->epoch - 1, peers->timeout);
    GS_CHECK_LAUNCH();
  }
  int rc = launch_phase1(poses, peers->disps[me], intrinsics, disps_sens, targets, weights, eta, eta_rows, ii, jj, d, ws,
                         motion_only, true, st);
  if (rc) return rc;
  if (peers->system[me] != ws.sys)
    cudaMemcpyAsync(peers->system[me], ws.sys, ((size_t)d.n * d.n + d.n) * sizeof(double), cudaMemcpyDeviceToDevice, st);
  // (2) publish: my partial system of iteration `epoch` is complete
  if (W > 1) {
    PeerRows rows{};
    rows.n = W;
    for (int r = 0; r < W; ++r) rows.p[r] = reinterpret_cast<float*>(peers->flags[r]);
    ba_peer_signal_kernel<<<1, 32, 0, st>>>(rows, me, peers->epoch);
    GS_CHECK_LAUNCH();
  }
  return GOSLAM_OK;
}

int goslam_ba_phase2_peers(float* poses, int N, int num, int ht, int wd, int t0, int t1, float lm, float ep,
                           int motion_only, int owner_lo, int owner_hi, const goslam_ba_peers* peers, float* dx_out,
                           float* dz_out, int* status_out, void* workspace, size_t workspace_bytes, void* stream) {
  BaDims d;
  if (!make_dims(N, num, ht, wd, t0, t1, &d) || !peers_ok(peers)) return GOSLAM_EINVAL;
  if (d.P == 0) return GOSLAM_OK;
  BaWs ws;
  const size_t need = ba_layout(d, workspace, workspace_bytes, &ws);
  if (workspace == nullptr || need > workspace_bytes) return GOSLAM_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int W = peers->world, me = peers->rank;
  SysSrc src{};
  src.n = W;
  for (int r = 0; r < W; ++r) src.p[r] = peers->system[r];
  src.flags = peers->flags[me]; src.epoch = peers->epoch; src.timeout = peers->timeout;
  PeerRows rows{};
  rows.n = W;
  for (int r = 0; r < W; ++r) rows.p[r] = peers->disps[r];
  const int rc = launch_phase2(poses, peers->disps[me], src, d, ws, lm, ep, motion_only, owner_lo, owner_hi, dx_out, dz_out,
                               status_out, st, rows);
  if (rc) return rc;
  if (W > 1) {
    PeerRows frows{};
    frows.n = W;
    for (int r = 0; r < W; ++r) frows.p[r] = reinterpret_cast<float*>(peers->flags[r]);
    ba_peer_signal_kernel<<<1, 32, 0, st>>>(frows, W + me, peers->epoch);
    GS_CHECK_LAUNCH();
  }
  return GOSLAM_OK;
}

int goslam_ba_peers_wait(const goslam_ba_peers* peers, void* stream) {
  if (!peers_ok(peers)) return GOSLAM_EINVAL;
  if (peers->world > 1) {
    ba_peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(peers->flags[peers->rank] + peers->world, peers->world,
                                                            peers->epoch, peers->timeout);
    GS_CHECK_LAUNCH();
  }
  return GOSLAM_OK;
}

int goslam_peer_alloc(size_t bytes, void** ptr, void* handle_out) {
  if (!ptr || !handle_out || bytes == 0) return GOSLAM_EINVAL;
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, bytes);
  if (e == cudaSuccess) e = cudaMemset(q, 0, bytes);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, q);
  if (e != cudaSuccess) { gs_note_cuda_error(e); if (q) cudaFree(q); return GOSLAM_ELAUNCH; }
  memcpy(handle_out, &h, sizeof(h));
  *ptr = q;
  return GOSLAM_OK;
}

int goslam_peer_free(void* ptr) {
  if (!ptr) return GOSLAM_EINVAL;
  const cudaError_t e = cudaFree(ptr);
  if (e != cudaSuccess) { gs_note_cuda_error(e); return GOSLAM_ELAUNCH; }
  return GOSLAM_OK;
}

int goslam_ipc_open(const void* handle, void** ptr) {
  if (!handle || !ptr) return GOSLAM_EINVAL;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  const cudaError_t e = cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) { gs_note_cuda_error(e); return GOSLAM_ELAUNCH; }
  return GOSLAM_OK;
}

int goslam_ipc_close(void* ptr) {
  if (!ptr) return GOSLAM_EINVAL;
  const cudaError_t e = cudaIpcCloseMemHandle(ptr);
  if (e != cudaSuccess) { gs_note_cuda_error(e); return GOSLAM_ELAUNCH; }
  return GOSLAM_OK;
}

}  // extern "C"
