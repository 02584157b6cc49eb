// Fused E-step / M-step of the MMSBM EM iteration for sm_100a.
//
// Replaces update_coefficients (src/kernels_numpy.py:43-79) + normalize_with_d x2 +
// normalize_with_self (src/expectation_maximization.py:118-155), i.e. the loop body of
// src/mmsbm.py:244-250, for S runs at once.  The omega[N,K,L] tensor of the reference is
// never formed.  omega is rank-1 in (k,l) once the rating r is fixed, so for a segment
// that fixes one side ("owner": a user in the by-user pass, an item in the by-item pass)
//
//     w_r[b]   = sum_a own[a] P[a][b][r]                      (once per segment)   [1]
//     S_n      = sum_b w_r[b] nbr_n[b]                        (per rating: one gathered row)
//     g_r[b]  += nbr_n[b] / max(S_n, eps)                     (per rating)         [2]
//     n_own[a] = own[a] * sum_{r,b} P[a][b][r] g_r[b]         (once per segment)   [3]
//     n_pr[a][b][r] = P[a][b][r] * sum_segments own[a] g_r[b] (rank-1 per segment) [4]
//
// which is the reference's sum reassociated (agreement ~1e-15 relative, tests/test_em_gpu.py).
//
// Kernels of one iteration (all runs in grid.y, run-major so one run's tables stay in L2):
//   prep_p_kernel        P in the two operand layouts of each side
//   interleave_runs_kernel  theta / eta rows of run groups side by side (pairs; six runs for eta
//                        rows of 20 doubles): a warp of the hot kernel serves a group of runs and
//                        gathers one contiguous row per rating
//   row_w_kernel         [1] for every user and item: W = own x Pw.  A lane owns a row, P sits in
//                        shared memory and every read of it is a warp broadcast
//                        (small_gemm_kernel: tiled fallback for row strides > 32 doubles)
//   segment_pass_kernel  [2] THE HOT KERNEL (segment_pass.cuh): one warp per piece of a segment
//                        streams its ratings; per rating it moves one neighbour row (8*NB bytes,
//                        one 256-bit load per lane of a group of G lanes) and 4 bytes of index.
//                        w comes from W via cp.async (prefetched one piece ahead), g overwrites W
//                        in place.  Pieces are claimed from a launch-wide queue by persistent
//                        CTAs (large problems) or from a per-CTA range of pieces (small ones).  Segments longer than MMSBM_PIECE_LEN ratings are cut into
//                        pieces by the work schedule built with the index (graph_build.cu); their
//                        partial g rows are added in piece order by segment_fixup_kernel
//   row_n_kernel         [3] n_own = (G x Pn) o own / max(deg,1)   (normalisation fused)
//   pr_accumulate_kernel [4] block-private register accumulators over a slab of segments
//   pr_finalize_kernel   fixed-order reduce over slabs, x P, normalise over ratings
// No atomics on data, every sum has a fixed order: results are bit-reproducible.
#include <stdlib.h>

#include "common.cuh"
#include "em_internal.cuh"
#include "segment_pass.cuh"

namespace mmsbm {

constexpr int kPrThreads = 128;
constexpr int kPrBatch = 16;    // segments staged per smem batch
constexpr int kGemmThreads = 256;
constexpr int kGemmBK = 32;     // k-slab of the small GEMM (lower when a streamed slab of B does not fit)
constexpr int kGemmTR = 4;      // rows per thread tile of the small GEMM

// g rows of long segments: add the partial rows of their pieces in piece order
__global__ void __launch_bounds__(128) segment_fixup_kernel(const SegArgs A) {
  const int run = blockIdx.y, RNB = A.R * A.NBp;
  const int n_long = __ldg(A.sched + 2);
  const int32_t* long_seg = A.sched + 4 + 3 * A.pmax;
  const int32_t* long_slot0 = long_seg + A.lmax;
  for (int li = blockIdx.x; li < n_long; li += gridDim.x) {
    const int sg = __ldg(long_seg + li), s0 = __ldg(long_slot0 + li), s1 = __ldg(long_slot0 + li + 1);
    MMSBM_DEV_CHECK(sg >= 0 && sg < A.nseg && s0 >= 0 && s0 < s1 && s1 <= A.smax);
    const double* src = A.partial + ((size_t)run * A.smax + s0) * RNB;
    double* dst = A.wg + ((size_t)run * A.nseg + sg) * RNB;
    for (int o = threadIdx.x; o < RNB; o += blockDim.x) {
      double acc = 0.0;
      for (int k = 0; k < s1 - s0; ++k) acc += src[(size_t)k * RNB + o];
      dst[o] = acc;
    }
  }
}

// ---- rows of run groups interleaved: dst[grp][row0 + id][j][ld] <- src[gs*grp + j][id][ld], j < gs,
//      for the groups [group0, group0 + groups); src holds n_src rows per run, dst n_dst rows per
//      group (n_dst > n_src when a rank fills its slice of a table that spans all ranks) ------
__global__ void interleave_runs_kernel(const double* __restrict__ src, double* __restrict__ dst, int n_src,
                                       int n_dst, int row0, int ld, int group0, int groups, int gs) {
  const int c4 = ld >> 2;
  const size_t total = (size_t)groups * n_src * gs * c4;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int c = (int)(t % c4);
  const int j = (int)((t / c4) % gs);
  const size_t rest = t / c4 / gs;
  const int id = (int)(rest % n_src);
  const size_t p = group0 + rest / n_src;
  const double4_t v = ldg256(src + (((size_t)(gs * p + j) * n_src + id) * ld + 4 * c));
  stg256(dst + (((p * n_dst + row0 + id) * gs + j) * ld + 4 * c), v);
}

// ---- P in operand layout -------------------------------------------------------------------
// For a side with owner dim NA (stride lda), neighbour dim NB (stride NBp), RNB = R*NBp and
// o = r*NBp + b:   Pw[a][o] (lda x RNB)   Pn[o][a] (RNB x lda),  zero in every padded slot.
// user side: a=k, b=l;  item side: a=l, b=k.  One thread per padded (k,l,r).
__global__ void prep_p_kernel(const double* pr, int K, int L, int R, int ldk, int ldl, double* pw_u,
                              double* pn_u, double* pw_i, double* pn_i) {
  const int run = blockIdx.y;
  const int total = ldk * ldl * R;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int r = t % R, kl = t / R, lp = kl % ldl, kp = kl / ldl;
  double v = 0.0;
  if (kp < K && lp < L) v = __ldg(pr + (((size_t)run * K + kp) * L + lp) * R + r);
  const size_t base = (size_t)run * total;
  const int rnb_u = R * ldl, rnb_i = R * ldk;
  pw_u[base + (size_t)kp * rnb_u + r * ldl + lp] = v;
  pn_u[base + (size_t)(r * ldl + lp) * ldk + kp] = v;
  pw_i[base + (size_t)lp * rnb_i + r * ldk + kp] = v;
  pn_i[base + (size_t)(r * ldk + kp) * ldl + lp] = v;
}

// ---- C[M x N] = A[M x Kd] . B[Kd x N] for tall-skinny fp64 problems (N, Kd <= ~1k) ------------
// Persistent CTAs: B is staged in shared memory once, then each CTA walks row tiles; one 4x4
// output tile per thread (rg row groups x N/4 column groups), A in k-slabs of g.bk rows (B too, when
// it does not fit shared memory whole).  Every thread adds its products in increasing k whatever
// the slab height, so the height does not change the result.  EPI: C = C o own / max(deg,1).
// fp64 FMA pipe, no tensor cores (B200 DMMA is no faster than the vector pipe and the path is not GEMM-bound).
struct GemmArgs {
  const double* A;      // [S][M][lda]
  const double* B;      // [S][Kd][N]
  double* C;            // [S][M][N]
  const double* own;    // EPI: [S][M][N]
  const int32_t* deg;   // EPI: [M]
  int M, N, Kd, lda, rg, normalize;
  int b_resident;       // whole B staged once (fits shared memory) or one k-slab at a time
  int bk;               // k-slab height: a multiple of 4, kGemmBK unless a slab of B would not fit
};

template <bool EPI>
__global__ void __launch_bounds__(kGemmThreads) small_gemm_kernel(const GemmArgs g) {
  constexpr int TR = kGemmTR;                  // rows of the register tile (columns: 4)
  extern __shared__ __align__(32) unsigned char smem_raw[];
  const int BM = TR * g.rg, AS = g.bk + 2;
  double* Bs = reinterpret_cast<double*>(smem_raw);          // [Kd][N] whole B, or [bk][N] slab
  double* As = Bs + (size_t)(g.b_resident ? g.Kd : g.bk) * g.N;   // [BM][AS] k-slab of a row tile
  const int run = blockIdx.y;
  const int ncg = g.N >> 2, half = g.N >> 1;
  const int rgid = threadIdx.x / ncg, cg = threadIdx.x - rgid * ncg;
  const bool active = rgid < g.rg;
  const double* A = g.A + (size_t)run * g.M * g.lda;
  const double2* B2 = reinterpret_cast<const double2*>(g.B + (size_t)run * g.Kd * g.N);
  double2* Bs2 = reinterpret_cast<double2*>(Bs);
  if (g.b_resident)
    for (int t = threadIdx.x; t < (g.Kd * g.N) >> 1; t += kGemmThreads) Bs2[t] = __ldg(B2 + t);
  const int n_tiles = (g.M + BM - 1) / BM;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * BM;
    double acc[TR][4];
#pragma unroll
    for (int i = 0; i < TR; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;

    for (int k0 = 0; k0 < g.Kd; k0 += g.bk) {
      const int bk = min(g.bk, g.Kd - k0);             // multiple of 4
      const int bk2 = bk >> 1;
      __syncthreads();
      for (int t = threadIdx.x; t < BM * bk2; t += kGemmThreads) {   // 128-bit staging of the A slab
        const int m = t / bk2, p2 = t - m * bk2;
        double2 v = make_double2(0.0, 0.0);
        if (row0 + m < g.M) v = __ldg(reinterpret_cast<const double2*>(A + (size_t)(row0 + m) * g.lda + k0) + p2);
        *reinterpret_cast<double2*>(As + m * AS + 2 * p2) = v;
      }
      if (!g.b_resident)
        for (int t = threadIdx.x; t < (bk * g.N) >> 1; t += kGemmThreads)
          Bs2[t] = __ldg(B2 + (((size_t)k0 * g.N) >> 1) + t);
      __syncthreads();
      if (active) {
        // thread tile: rows TR*rgid.., columns {2cg, 2cg+1, N/2+2cg, N/2+2cg+1}: consecutive
        // threads read consecutive 16-byte pieces of a B row (no bank conflicts); the A reads of
        // a warp are (nearly) uniform, i.e. broadcasts
        const double* ap = As + (size_t)(TR * rgid) * AS;
        const double* bp = Bs + (size_t)(g.b_resident ? k0 : 0) * g.N + 2 * cg;
        for (int kk = 0; kk < bk; kk += 2) {
          const double2 b00 = *reinterpret_cast<const double2*>(bp + (size_t)kk * g.N);
          const double2 b01 = *reinterpret_cast<const double2*>(bp + (size_t)kk * g.N + half);
          const double2 b10 = *reinterpret_cast<const double2*>(bp + (size_t)(kk + 1) * g.N);
          const double2 b11 = *reinterpret_cast<const double2*>(bp + (size_t)(kk + 1) * g.N + half);
#pragma unroll
          for (int i = 0; i < TR; ++i) {
            const double2 a = *reinterpret_cast<const double2*>(ap + i * AS + kk);
            acc[i][0] = fma(a.x, b00.x, acc[i][0]); acc[i][1] = fma(a.x, b00.y, acc[i][1]);
            acc[i][2] = fma(a.x, b01.x, acc[i][2]); acc[i][3] = fma(a.x, b01.y, acc[i][3]);
            acc[i][0] = fma(a.y, b10.x, acc[i][0]); acc[i][1] = fma(a.y, b10.y, acc[i][1]);
            acc[i][2] = fma(a.y, b11.x, acc[i][2]); acc[i][3] = fma(a.y, b11.y, acc[i][3]);
          }
        }
      }
    }
    if (active) {
#pragma unroll
      for (int i = 0; i < TR; ++i) {
        const int m = row0 + TR * rgid + i;
        if (m >= g.M) continue;
        const size_t off = ((size_t)run * g.M + m) * g.N + 2 * cg;
        double2 v0 = make_double2(acc[i][0], acc[i][1]), v1 = make_double2(acc[i][2], acc[i][3]);
        if (EPI) {
          const double2 o0 = __ldg(reinterpret_cast<const double2*>(g.own + off));
          const double2 o1 = __ldg(reinterpret_cast<const double2*>(g.own + off + half));
          v0.x *= o0.x; v0.y *= o0.y; v1.x *= o1.x; v1.y *= o1.y;
          if (g.normalize) {
            const double d = (double)max(__ldg(g.deg + m), 1);
            v0.x = v0.x / d; v0.y = v0.y / d; v1.x = v1.x / d; v1.y = v1.y / d;
          }
        }
        *reinterpret_cast<double2*>(g.C + off) = v0;
        *reinterpret_cast<double2*>(g.C + off + half) = v1;
      }
    }
  }
}

// ---- lane-per-row variants of the two contractions (row strides <= 32 doubles) ---------------
// A lane owns one segment: its own-row (w) or its accumulators (n) live in registers, the P
// table sits in shared memory and every read of it is a warp-wide broadcast (one wavefront),
// so the kernels need no barriers and little LSU bandwidth; HBM traffic is the W / G rows.
constexpr int kRowThreads = 256;

// ROWS rows per lane: every 32-byte read of P from shared memory (a warp broadcast) feeds
// 4*ROWS DFMAs, so with two rows the fp64 pipe, not the shared-memory pipe, sets the pace.
template <int LD, int ROWS>
__global__ void __launch_bounds__(kRowThreads) row_w_kernel(const double* __restrict__ own,
                                                            const double* __restrict__ pw,
                                                            double* __restrict__ W, int M, int RNB) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  double* Ps = reinterpret_cast<double*>(smem_raw);          // [LD][RNB]
  const int run = blockIdx.y;
  {
    const double2* src = reinterpret_cast<const double2*>(pw + (size_t)run * LD * RNB);
    double2* dst = reinterpret_cast<double2*>(Ps);
    for (int t = threadIdx.x; t < (LD * RNB) >> 1; t += kRowThreads) dst[t] = __ldg(src + t);
  }
  __syncthreads();
  const double* own_run = own + (size_t)run * M * LD;
  double* w_run = W + (size_t)run * M * RNB;
  for (int m0 = blockIdx.x * (kRowThreads * ROWS) + threadIdx.x; m0 < M; m0 += gridDim.x * (kRowThreads * ROWS)) {
    double o[ROWS][LD];
    int mr[ROWS];
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      mr[j] = m0 + j * kRowThreads;
      const int mc = mr[j] < M ? mr[j] : m0;                 // rows past the end recompute row m0
#pragma unroll
      for (int c = 0; c < LD / 4; ++c) {
        const double4_t v = ldg256(own_run + (size_t)mc * LD + 4 * c);
        o[j][4 * c] = v.x; o[j][4 * c + 1] = v.y; o[j][4 * c + 2] = v.z; o[j][4 * c + 3] = v.w;
      }
    }
    for (int ob = 0; ob < RNB; ob += 4) {
      double4_t acc[ROWS];
#pragma unroll
      for (int j = 0; j < ROWS; ++j) acc[j] = double4_t{0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int a = 0; a < LD; ++a) {
        const double4_t p = lds32(Ps + a * RNB + ob);
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
          acc[j].x = fma(o[j][a], p.x, acc[j].x); acc[j].y = fma(o[j][a], p.y, acc[j].y);
          acc[j].z = fma(o[j][a], p.z, acc[j].z); acc[j].w = fma(o[j][a], p.w, acc[j].w);
        }
      }
#pragma unroll
      for (int j = 0; j < ROWS; ++j)
        if (mr[j] < M) stg256(w_run + (size_t)mr[j] * RNB + ob, acc[j]);
    }
  }
}

// PF chunks (32 bytes each) of the G row are loaded back to back before any of them is used: a lane
// then has PF loads in flight instead of one, which is what the HBM stream of this kernel needs
// (lane-per-row rows are 800 bytes apart, so memory-level parallelism has to come from depth).
template <int LD, int ROWS, int PF>
__global__ void __launch_bounds__(kRowThreads) row_n_kernel(const double* __restrict__ G,
                                                            const double* __restrict__ pn,
                                                            const double* __restrict__ own,
                                                            const int32_t* __restrict__ deg,
                                                            double* __restrict__ out, int M, int RNB,
                                                            int normalize, const RowPublish pub) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  double* Ps = reinterpret_cast<double*>(smem_raw);          // [RNB][LD]
  const int run = blockIdx.y;
  // the gather table (if any) that serves this run: the new rows are stored there too
  double* pdst = nullptr;
  int pgs = 1, pj = 0;
  size_t pgrp = 0;
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    if (pub.dst[t] != nullptr && run >= pub.gs[t] * pub.group0[t] && run < pub.gs[t] * (pub.group0[t] + pub.groups[t])) {
      pdst = pub.dst[t]; pgs = pub.gs[t]; pgrp = (size_t)(run / pub.gs[t]); pj = run % pub.gs[t];
    }
  }
  {
    const double2* src = reinterpret_cast<const double2*>(pn + (size_t)run * LD * RNB);
    double2* dst = reinterpret_cast<double2*>(Ps);
    for (int t = threadIdx.x; t < (LD * RNB) >> 1; t += kRowThreads) dst[t] = __ldg(src + t);
  }
  __syncthreads();
  const double* g_run = G + (size_t)run * M * RNB;
  const double* own_run = own + (size_t)run * M * LD;
  double* out_run = out + (size_t)run * M * LD;
  for (int m0 = blockIdx.x * (kRowThreads * ROWS) + threadIdx.x; m0 < M; m0 += gridDim.x * (kRowThreads * ROWS)) {
    double acc[ROWS][LD];
    int mr[ROWS];
    const double* grow[ROWS];
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      mr[j] = m0 + j * kRowThreads;
      grow[j] = g_run + (size_t)(mr[j] < M ? mr[j] : m0) * RNB;   // rows past the end recompute row m0
#pragma unroll
      for (int a = 0; a < LD; ++a) acc[j][a] = 0.0;
    }
    for (int ob0 = 0; ob0 < RNB; ob0 += 4 * PF) {             // RNB is a multiple of 4 * PF (host checks)
      double4_t gq[ROWS][PF];
#pragma unroll
      for (int j = 0; j < ROWS; ++j)
#pragma unroll
        for (int p = 0; p < PF; ++p) gq[j][p] = ldg256(grow[j] + ob0 + 4 * p);
#pragma unroll
      for (int p = 0; p < PF; ++p) {
        const int ob = ob0 + 4 * p;
        double gv[ROWS][4];
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
          gv[j][0] = gq[j][p].x; gv[j][1] = gq[j][p].y; gv[j][2] = gq[j][p].z; gv[j][3] = gq[j][p].w;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int c = 0; c < LD / 4; ++c) {
            const double4_t pv = lds32(Ps + (ob + i) * LD + 4 * c);
#pragma unroll
            for (int j = 0; j < ROWS; ++j) {
              acc[j][4 * c] = fma(gv[j][i], pv.x, acc[j][4 * c]);         acc[j][4 * c + 1] = fma(gv[j][i], pv.y, acc[j][4 * c + 1]);
              acc[j][4 * c + 2] = fma(gv[j][i], pv.z, acc[j][4 * c + 2]); acc[j][4 * c + 3] = fma(gv[j][i], pv.w, acc[j][4 * c + 3]);
            }
          }
        }
      }
    }
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
      if (mr[j] >= M) continue;
      double d = 1.0;
      if (normalize) d = (double)max(__ldg(deg + mr[j]), 1);
#pragma unroll
      for (int c = 0; c < LD / 4; ++c) {
        const double4_t ov = ldg256(own_run + (size_t)mr[j] * LD + 4 * c);
        double4_t v{acc[j][4 * c] * ov.x, acc[j][4 * c + 1] * ov.y, acc[j][4 * c + 2] * ov.z, acc[j][4 * c + 3] * ov.w};
        if (normalize) { v.x = v.x / d; v.y = v.y / d; v.z = v.z / d; v.w = v.w / d; }
        stg256(out_run + (size_t)mr[j] * LD + 4 * c, v);
        if (pdst) stg256(pdst + (((pgrp * pub.n_all + pub.row0 + mr[j]) * pgs + pj) * LD + 4 * c), v);
      }
    }
  }
}

// ---- n_pr: Acc[a][r][b] = sum_seg own[seg][a] g[seg][r][b], per-CTA private accumulators,
//      one partial per slab, reduced in fixed order by pr_finalize_kernel -------------------
struct PrArgs {
  const double* own;   // [S][nseg][lda]
  const double* g;     // [S][nseg][RNB]
  double* partial;     // [S][kPrSlabs][NA*RNB]
  int nseg, NA, lda, RNB;
};

__global__ void __launch_bounds__(kPrThreads) pr_accumulate_kernel(const PrArgs A) {
  // 4x4 register tiles (4 owner indices x 4 consecutive (r,b) outputs): per staged segment a
  // thread reads two 32-byte vectors from shared memory for 16 FMAs
  extern __shared__ __align__(32) unsigned char smem_raw[];
  double* own_s = reinterpret_cast<double*>(smem_raw);   // [kPrBatch][lda]
  double* g_s = own_s + kPrBatch * A.lda;                // [kPrBatch][RNB]
  const int run = blockIdx.y, slab = blockIdx.x;
  const int per = (A.nseg + kPrSlabs - 1) / kPrSlabs;
  const int s0 = slab * per, s1 = min(s0 + per, A.nseg);
  const int nout = A.NA * A.RNB;
  const int ta = A.lda >> 2, tb = A.RNB >> 2, n_tiles = ta * tb;
  const double* own_run = A.own + (size_t)run * A.nseg * A.lda;
  const double* g_run = A.g + (size_t)run * A.nseg * A.RNB;
  double* dst = A.partial + ((size_t)run * kPrSlabs + slab) * nout;

  for (int tile0 = 0; tile0 < n_tiles; tile0 += kPrThreads) {
    const int tile = tile0 + threadIdx.x;
    const bool on = tile < n_tiles;
    const int a0 = on ? 4 * (tile / tb) : 0, b0 = on ? 4 * (tile % tb) : 0;
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int k = 0; k < 4; ++k) acc[i][k] = 0.0;
    for (int c0 = s0; c0 < s1; c0 += kPrBatch) {
      const int nb = min(kPrBatch, s1 - c0);
      __syncthreads();
      {   // rows of both tables are whole 16-byte pieces
        const double2* src = reinterpret_cast<const double2*>(own_run + (size_t)c0 * A.lda);
        double2* d2 = reinterpret_cast<double2*>(own_s);
        for (int t = threadIdx.x; t < (nb * A.lda) >> 1; t += kPrThreads) d2[t] = __ldg(src + t);
        src = reinterpret_cast<const double2*>(g_run + (size_t)c0 * A.RNB);
        d2 = reinterpret_cast<double2*>(g_s);
        for (int t = threadIdx.x; t < (nb * A.RNB) >> 1; t += kPrThreads) d2[t] = __ldg(src + t);
      }
      __syncthreads();
      if (on) {
        for (int sg = 0; sg < nb; ++sg) {
          const double4_t o = lds32(own_s + sg * A.lda + a0);
          const double4_t g = lds32(g_s + sg * A.RNB + b0);
          const double ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            acc[i][0] = fma(ov[i], g.x, acc[i][0]); acc[i][1] = fma(ov[i], g.y, acc[i][1]);
            acc[i][2] = fma(ov[i], g.z, acc[i][2]); acc[i][3] = fma(ov[i], g.w, acc[i][3]);
          }
        }
      }
    }
    if (on) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (a0 + i < A.NA)
          stg256(dst + (size_t)(a0 + i) * A.RNB + b0, double4_t{acc[i][0], acc[i][1], acc[i][2], acc[i][3]});
    }
  }
}

struct PrFinArgs {
  const double* partial;  // [S][kPrSlabs][NA*RNB]
  const double* pr;       // [S][K][L][R]
  double* pr_out;         // [S][K][L][R]
  int K, L, R, NA, NBp, transposed, normalize;
};

// One block per (owner index a, run): n_pr[a][b][r] = P * sum over slabs of Acc, then every
// (k,l) row over r is divided by its sum (a sum that is exactly zero divides by one,
// expectation_maximization.py:154).  Warp w adds its share of the slabs for 32 consecutive
// outputs at a time (coalesced), the warps' sums are added in warp order: fixed order throughout.
constexpr int kFinWarps = 8;
__global__ void __launch_bounds__(kFinWarps * 32) pr_finalize_kernel(const PrFinArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int run = blockIdx.y, a = blockIdx.x;
  const int RNB = A.R * A.NBp, nout = A.NA * RNB;
  double* part_s = reinterpret_cast<double*>(smem_raw);      // [kFinWarps][RNB]
  double* tot_s = part_s + kFinWarps * RNB;                  // [RNB]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double* part = A.partial + (size_t)run * kPrSlabs * nout + (size_t)a * RNB;
  constexpr int per = kPrSlabs / kFinWarps;
  for (int o = lane; o < RNB; o += 32) {
    double acc = 0.0;
#pragma unroll 4
    for (int s = warp * per; s < (warp + 1) * per; ++s) acc += part[(size_t)s * nout + o];
    part_s[warp * RNB + o] = acc;
  }
  __syncthreads();
  for (int o = threadIdx.x; o < RNB; o += blockDim.x) {
    double acc = 0.0;
    for (int w = 0; w < kFinWarps; ++w) acc += part_s[w * RNB + o];
    tot_s[o] = acc;
  }
  __syncthreads();
  const int NB = A.transposed ? A.K : A.L;
  for (int b = threadIdx.x; b < NB; b += blockDim.x) {
    const int k = A.transposed ? b : a, l = A.transposed ? a : b;
    const size_t kl = (size_t)k * A.L + l;
    const double* prs = A.pr + ((size_t)run * A.K * A.L + kl) * A.R;
    double* dst = A.pr_out + ((size_t)run * A.K * A.L + kl) * A.R;
    double tot = 0.0;
    for (int r = 0; r < A.R; ++r) {
      const double v = tot_s[r * A.NBp + b] * prs[r];
      dst[r] = v;
      tot += v;
    }
    if (A.normalize) {
      const double d = (tot == 0.0) ? 1.0 : tot;
      for (int r = 0; r < A.R; ++r) dst[r] = dst[r] / d;
    }
  }
}

// post-all-reduce epilogue (rating-sharded runs)
__global__ void finalize_eta_kernel(double* eta, const int32_t* deg, int n_items, int ldl, int L,
                                    size_t total) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  int col = (int)(t % ldl);
  size_t row = t / ldl;
  int item = (int)(row % n_items);
  if (col < L) eta[t] = eta[t] / (double)max(__ldg(deg + item), 1);
}

__global__ void finalize_pr_kernel(double* pr, int KL_total, int R) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= KL_total) return;
  double* row = pr + (size_t)t * R;
  double tot = 0.0;
  for (int r = 0; r < R; ++r) tot += row[r];
  const double d = (tot == 0.0) ? 1.0 : tot;
  for (int r = 0; r < R; ++r) row[r] = row[r] / d;
}

// ------------------------------------------------------------------------------------------
struct PassShape { int G, CH, UN, MINB; };

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

// multiprocessors of the current device (148 on a B200), cached per device ordinal
int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// NCH 32-byte chunks per row are spread over G lanes x CH chunks per lane with G <= 8 (three
// shuffle levels per rating at most); UN steps in flight; MINB CTAs per SM the kernel is
// compiled for.  Defaults from the sweeps recorded in DESIGN.md section 5.
static PassShape choose_shape(int NBp) {
  const int NCH = NBp / 4;
  int CH = 8;
  for (int c = 1; c <= 8; c *= 2) {
    if ((NCH + c - 1) / c <= 8) { CH = c; break; }
  }
  const int G = (NCH + CH - 1) / CH;
  PassShape sh{G, CH, 1, 1};   // CH == 1 implies NBp == 4*G (the kernel relies on it)
  // three row loads in flight per warp, 3 CTAs/SM: best of the UN x MINB sweep on both passes
  // (four loads spill at 80 registers, 128 registers cost a third of the resident warps)
  if (CH == 1) { sh.UN = (G == 1) ? 1 : (G == 2) ? 2 : 3; sh.MINB = 3; }   // UN * (32 / G) <= 32
  else if (CH == 2) { sh.UN = 1; sh.MINB = 3; }
  return sh;
}

// Pieces per CTA, a multiple of the warps per CTA (the warps claim pieces dynamically; with 9
// pieces for 8 warps the CTA would last two piece times).  Two rules from the sweep in
// profiles/r1_spc_sweep.txt: about 6k ratings of work per CTA -- short segments want several per
// warp to even out, long pieces want one per warp so that the last wave of CTAs is short -- and
// at least ~6 CTAs per resident slot (148 SMs x 3) whatever the problem size.
static int segs_per_cta_for(int64_t pmax, int64_t n_ratings, int grid_y) {
  const double avg_piece = (double)(n_ratings > 0 ? n_ratings : 1) / (double)(pmax > 0 ? pmax : 1);
  int64_t spc = ((int64_t)(6144.0 / (avg_piece > 1.0 ? avg_piece : 1.0)) + kWarps / 2) / kWarps * kWarps;
  const int64_t fill = pmax * grid_y / (sm_count() * 3 * 6) / kWarps * kWarps;
  if (spc > fill) spc = fill;
  if (spc < kWarps) spc = kWarps;               // one piece per warp at least
  if (spc > 64) spc = 64;
  return (int)spc;
}

// pairs of runs per warp whenever there are at least two runs, a lane holds one chunk and the
// w rows of a pair fit shared memory
static bool pairs_enabled(int NBp, int R, int n_runs) {
  return n_runs >= 2 && NBp <= 32 && seg_smem_bytes(R, NBp, 2) <= kMaxSmemBytes;
}

// grid.x of a segment pass.  The piece count lives on the device, so the grid is sized for its upper
// bound (warps past it exit).  With launch-wide claiming (a.counters) the CTAs are persistent: as
// many as stay resident (148 SMs x CTAs per SM), one starting piece per warp at least.
static int g_reserved_ctas = 0;
void set_reserved_ctas(int n) { g_reserved_ctas = n > 0 ? n : 0; }

static unsigned grid_x_for(const SegArgs& a, int ctas_per_sm) {
  if (!a.counters) return (unsigned)((a.pmax + a.segs_per_cta - 1) / a.segs_per_cta);
  int64_t resident = (int64_t)sm_count() * ctas_per_sm - g_reserved_ctas;
  if (resident < 1) resident = 1;
  const int64_t want = (a.pmax + kWarps - 1) / kWarps;
  return (unsigned)(want < resident ? want : resident);
}

// six runs per warp: rows of exactly 20 doubles (5-lane groups, 30 of 32 lanes), at least six runs,
// and the w rows of six runs fit shared memory (R <= 30)
static bool hexa_enabled(int NBp, int R, int n_runs) {
  return n_runs >= 6 && NBp == 20 && seg_smem_bytes(R, NBp, 6) <= kMaxSmemBytes;
}

RunPlan plan_runs(int NBp, int R, int n_runs, bool hexa_table) {
  RunPlan p{0, 0, 0, 0};
  if (hexa_table && hexa_enabled(NBp, R, n_runs)) p.hexas = n_runs / 6;
  p.single_from = 6 * p.hexas;
  if (pairs_enabled(NBp, R, n_runs - p.single_from)) {
    p.pairs = (n_runs - p.single_from) / 2;
    p.pair_group0 = p.single_from / 2;            // pairs are numbered over all runs (6 | single_from)
    p.single_from += 2 * p.pairs;
  }
  return p;
}

static int launch_segment_pass_impl(SegArgs a, const double* nbr_pairs, const double* nbr_hexa,
                                    int64_t n_ratings, int n_runs, cudaStream_t st) {
  const PassShape sh = choose_shape(a.NBp);
  const RunPlan plan = plan_runs(a.NBp, a.R, n_runs, nbr_hexa != nullptr);
  const int single_from = plan.single_from;      // runs [single_from, n_runs) go one run per warp
  if (plan.hexas > 0) {
    const int hexas = plan.hexas;
    SegArgs p = a;
    p.nbr = nbr_hexa;
    p.run_base = 0;
    p.grp_base = 0;
    p.segs_per_cta = segs_per_cta_for(a.pmax, n_ratings, hexas);
    const unsigned gx = grid_x_for(p, 3);
    if (p.counters) a.counters += hexas;         // the next launch of this pass gets its own counters
    const size_t smem = seg_smem_bytes(a.R, a.NBp, 6);   // fits: plan_runs checked it
    const int rc = launch_segment_pass_hexa(p, sh.G, 3, 3, dim3(gx, hexas), smem, st);
    if (rc) {
      if (rc == MMSBM_ERANGE) set_error("no six-run segment-pass variant for G=%d", sh.G);
      return rc;
    }
    if (single_from == n_runs && plan.pairs == 0) return 0;
  }
  if (plan.pairs > 0) {
    MMSBM_REQUIRE(nbr_pairs, MMSBM_EINVAL, "segment pass: the table of run pairs is missing");
    const int pairs = plan.pairs;
    SegArgs p = a;
    p.nbr = nbr_pairs;
    p.run_base = 6 * plan.hexas;
    p.grp_base = plan.pair_group0;
    p.counters = a.counters;
    p.segs_per_cta = segs_per_cta_for(a.pmax, n_ratings, pairs);
    const int UN = (sh.G == 1) ? 2 : 3, MINB = 3;               // UN * (32 / 2G) <= 32
    const unsigned gx = grid_x_for(p, MINB);
    if (p.counters) a.counters += pairs;
    const size_t smem = seg_smem_bytes(a.R, a.NBp, 2);   // fits: plan_runs checked it
    const int rc = launch_segment_pass_pair(p, sh.G, UN, MINB, dim3(gx, pairs), smem, st);
    if (rc) {
      if (rc == MMSBM_ERANGE) set_error("no paired segment-pass variant for G=%d", sh.G);
      return rc;
    }
  }
  if (single_from == n_runs) return 0;
  a.run_base = single_from;
  a.segs_per_cta = segs_per_cta_for(a.pmax, n_ratings, n_runs - single_from);
  const unsigned gx = grid_x_for(a, sh.MINB);
  const dim3 grid(gx, n_runs - single_from);
  const size_t smem = seg_smem_bytes(a.R, a.NBp, 1);
  MMSBM_REQUIRE(smem <= kMaxSmemBytes, MMSBM_ERANGE,
                "segment pass needs %zu bytes of shared memory (R=%d, row stride %d)", smem, a.R, a.NBp);
  int rc;
  switch (sh.CH) {
    case 1: rc = launch_segment_pass_ch1(a, sh.G, sh.UN, sh.MINB, grid, smem, st); break;
    case 2: rc = launch_segment_pass_ch2(a, sh.G, sh.UN, sh.MINB, grid, smem, st); break;
    case 4: rc = launch_segment_pass_ch4(a, sh.G, sh.UN, sh.MINB, grid, smem, st); break;
    default: rc = launch_segment_pass_ch8(a, sh.G, sh.UN, sh.MINB, grid, smem, st); break;
  }
  if (rc == MMSBM_ERANGE) set_error("no segment-pass variant for G=%d CH=%d UN=%d", sh.G, sh.CH, sh.UN);
  return rc;
}

int launch_segment_pass_and_fixup(SegArgs a, const double* nbr_pairs, const double* nbr_hexa,
                                  int64_t n_ratings, int n_runs, cudaStream_t st, bool no_long_segments) {
  int rc = launch_segment_pass_impl(a, nbr_pairs, nbr_hexa, n_ratings, n_runs, st);
  if (rc) return rc;
  if (no_long_segments) return 0;               // the caller has read the schedule: nothing to add up
  const int64_t fix_ctas = 4 * sm_count();
  const unsigned gx = (unsigned)(a.lmax < fix_ctas ? a.lmax : fix_ctas);
  segment_fixup_kernel<<<dim3(gx, n_runs), 128, 0, st>>>(a);
  MMSBM_LAUNCH_CHECK("segment_fixup_kernel");
  return 0;
}

template <bool EPI>
static int launch_gemm(GemmArgs g, int n_runs, cudaStream_t st) {
  const int ncg = g.N / 4;
  MMSBM_REQUIRE(g.N % 4 == 0 && g.Kd % 4 == 0 && ncg >= 1 && ncg <= kGemmThreads, MMSBM_ERANGE,
                "small gemm: N=%d Kd=%d not supported (N <= 1024, multiples of 4)", g.N, g.Kd);
  int rg = kGemmThreads / ncg;
  if (rg > 32) rg = 32;
  g.rg = rg;
  const int BM = kGemmTR * rg;
  g.bk = kGemmBK;
  size_t smem = ((size_t)g.Kd * g.N + (size_t)BM * (g.bk + 2)) * 8;
  g.b_resident = smem <= 200 * 1024;
  if (!g.b_resident) {
    // streamed B: slabs of kGemmBK rows where they fit, otherwise the tallest multiple of 4 that does
    auto slab_bytes = [&](int bk) { return ((size_t)bk * g.N + (size_t)BM * (bk + 2)) * 8; };
    while (g.bk > 4 && slab_bytes(g.bk) > kMaxSmemBytes) g.bk -= 4;
    smem = slab_bytes(g.bk);
  }
  MMSBM_REQUIRE(smem <= kMaxSmemBytes, MMSBM_ERANGE,
                "small gemm needs %zu bytes of shared memory (K*L*R too large)", smem);
  auto kern = small_gemm_kernel<EPI>;
  MMSBM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int n_tiles = (g.M + BM - 1) / BM;
  int per_run = (sm_count() * 3 + n_runs - 1) / n_runs;      // ~3 persistent CTAs per SM in total
  if (per_run > n_tiles) per_run = n_tiles;
  if (per_run < 1) per_run = 1;
  kern<<<dim3(per_run, n_runs), kGemmThreads, smem, st>>>(g);
  MMSBM_LAUNCH_CHECK("small_gemm_kernel");
  return 0;
}

// dispatch of the two contractions: lane-per-row kernels for row strides <= 32, tiled GEMM beyond
int launch_w(const double* own, const double* pw, double* W, int M, int LD, int RNB, int n_runs,
             cudaStream_t st) {
  const size_t smem = (size_t)LD * RNB * 8;
#define MMSBM_ROW_W(LDv)                                                                        \
  if (LD == LDv && smem <= 200 * 1024) {                                                        \
    constexpr int kRows = (LDv <= 24) ? 2 : 1;   /* 2 x LD operand registers per lane */          \
    auto kern = row_w_kernel<LDv, kRows>;                                                       \
    const int per = kRowThreads * kRows;                                                        \
    const int gx = min((M + per - 1) / per, sm_count() * 2);                                    \
    MMSBM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<dim3(gx, n_runs), kRowThreads, smem, st>>>(own, pw, W, M, RNB);                      \
    MMSBM_LAUNCH_CHECK("row_w_kernel");                                                         \
    return 0;                                                                                   \
  }
  MMSBM_ROW_W(4) MMSBM_ROW_W(8) MMSBM_ROW_W(12) MMSBM_ROW_W(16) MMSBM_ROW_W(20) MMSBM_ROW_W(24)
  MMSBM_ROW_W(28) MMSBM_ROW_W(32)
#undef MMSBM_ROW_W
  GemmArgs g{own, pw, W, nullptr, nullptr, M, RNB, LD, LD, 0, 0, 0, kGemmBK};
  return launch_gemm<false>(g, n_runs, st);
}

int launch_n(const double* G, const double* pn, const double* own, const int32_t* deg, double* out,
             int M, int LD, int RNB, int normalize, int n_runs, cudaStream_t st, const RowPublish* publish) {
  const size_t smem = (size_t)LD * RNB * 8;
  RowPublish pub{};
  if (publish) pub = *publish;
  // one row per lane here: two rows cost occupancy (142 registers) and measured slower.  PF chunks
  // of the G row in flight per lane; PF must divide RNB / 4
  const int pf = (RNB / 4) % 5 == 0 ? 5 : (RNB / 4) % 2 == 0 ? 2 : 1;
#define MMSBM_ROW_N_GO(kern)                                                                    \
  {                                                                                             \
    const int gx = min((M + kRowThreads - 1) / kRowThreads, sm_count() * 2);                    \
    MMSBM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<dim3(gx, n_runs), kRowThreads, smem, st>>>(G, pn, own, deg, out, M, RNB, normalize, pub); \
    MMSBM_LAUNCH_CHECK("row_n_kernel");                                                         \
    return 0;                                                                                   \
  }
#define MMSBM_ROW_N(LDv)                                                                        \
  if (LD == LDv && smem <= 200 * 1024) {                                                        \
    if (pf == 5) MMSBM_ROW_N_GO((row_n_kernel<LDv, 1, 5>))                                      \
    if (pf == 2) MMSBM_ROW_N_GO((row_n_kernel<LDv, 1, 2>))                                      \
    MMSBM_ROW_N_GO((row_n_kernel<LDv, 1, 1>))                                                   \
  }
  MMSBM_ROW_N(4) MMSBM_ROW_N(8) MMSBM_ROW_N(12) MMSBM_ROW_N(16) MMSBM_ROW_N(20) MMSBM_ROW_N(24)
  MMSBM_ROW_N(28) MMSBM_ROW_N(32)
#undef MMSBM_ROW_N_GO
#undef MMSBM_ROW_N
  GemmArgs g{G, pn, out, own, deg, M, LD, RNB, RNB, 0, normalize, 0, kGemmBK};
  int rc = launch_gemm<true>(g, n_runs, st);
  if (rc || !publish) return rc;
  // the tiled path (a P table of more than 200 KB) writes `out` only: copy the new rows into the
  // gather tables afterwards
  for (int t = 0; t < 3; ++t)
    if (pub.dst[t] && (rc = launch_interleave(out, pub.dst[t], M, pub.n_all, pub.row0, LD, pub.group0[t],
                                              pub.groups[t], pub.gs[t], st)))
      return rc;
  return 0;
}

int launch_prep_p(const double* pr, int K, int L, int R, int ldk, int ldl, int n_runs, double* pw_u,
                  double* pn_u, double* pw_i, double* pn_i, cudaStream_t st) {
  const int total = ldk * ldl * R;
  prep_p_kernel<<<dim3((total + 255) / 256, n_runs), 256, 0, st>>>(pr, K, L, R, ldk, ldl, pw_u, pn_u, pw_i, pn_i);
  MMSBM_LAUNCH_CHECK("prep_p_kernel");
  return 0;
}

int launch_interleave(const double* src, double* dst, int n_src, int n_dst, int row0, int ld, int group0,
                      int groups, int gs, cudaStream_t st) {
  const size_t tot = (size_t)groups * n_src * gs * (ld / 4);
  if (tot == 0) return 0;
  interleave_runs_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(src, dst, n_src, n_dst, row0, ld,
                                                                        group0, groups, gs);
  MMSBM_LAUNCH_CHECK("interleave_runs_kernel");
  return 0;
}

int launch_pr(const double* own, const double* g, double* partial, const double* pr, double* pr_out,
              int nseg, int NA, int lda, int NBp, int K, int L, int R, int n_runs, bool transposed,
              bool normalize, cudaStream_t st) {
  PrArgs pa{};
  pa.own = own; pa.g = g; pa.partial = partial;
  pa.nseg = nseg; pa.NA = NA; pa.lda = lda; pa.RNB = R * NBp;
  const size_t smem = (size_t)kPrBatch * (pa.lda + pa.RNB) * 8;
  MMSBM_CUDA(cudaFuncSetAttribute(pr_accumulate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
  pr_accumulate_kernel<<<dim3(kPrSlabs, n_runs), kPrThreads, smem, st>>>(pa);
  MMSBM_LAUNCH_CHECK("pr_accumulate_kernel");
  PrFinArgs fa{};
  fa.partial = partial; fa.pr = pr; fa.pr_out = pr_out;
  fa.K = K; fa.L = L; fa.R = R; fa.NA = NA; fa.NBp = NBp;
  fa.transposed = transposed ? 1 : 0;
  fa.normalize = normalize ? 1 : 0;
  const size_t fin_smem = (size_t)(kFinWarps + 1) * R * NBp * 8;
  MMSBM_CUDA(cudaFuncSetAttribute(pr_finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
  pr_finalize_kernel<<<dim3(NA, n_runs), kFinWarps * 32, fin_smem, st>>>(fa);
  MMSBM_LAUNCH_CHECK("pr_finalize_kernel");
  return 0;
}

int launch_finalize_pr(double* pr, int kl_total, int R, cudaStream_t st) {
  finalize_pr_kernel<<<(kl_total + 127) / 128, 128, 0, st>>>(pr, kl_total, R);
  MMSBM_LAUNCH_CHECK("finalize_pr_kernel");
  return 0;
}

struct EmDims {
  int U, I, R, K, L, S, ldk, ldl, rnb_u, rnb_i;
  bool emit_items;   // the side with fewer segments carries the pr accumulation
  int nseg_e, NA_e, NBp_e;
  size_t p_elems, wg_u_elems, wg_i_elems, partial_elems, slots_u_elems, slots_i_elems;
  size_t th2_elems, et2_elems;   // theta / eta with the rows of run pairs interleaved
  size_t et6_elems;              // eta with the rows of groups of six runs interleaved (by-user pass)
  size_t ctr_elems;              // int32 piece counters: one per launch row (grid.y), both passes
  int64_t lmax, smax, pmax_u, pmax_i;
};

static EmDims em_dims(int64_t N, int U, int I, int R, int K, int L, int S) {
  EmDims d;
  d.U = U; d.I = I; d.R = R; d.K = K; d.L = L; d.S = S;
  d.ldk = row_stride(K); d.ldl = row_stride(L);
  d.rnb_u = R * d.ldl; d.rnb_i = R * d.ldk;
  d.emit_items = (I <= U);
  d.nseg_e = d.emit_items ? I : U;
  d.NA_e = d.emit_items ? L : K;
  d.NBp_e = d.emit_items ? d.ldk : d.ldl;
  d.p_elems = (size_t)S * d.ldk * d.ldl * R;
  d.wg_u_elems = (size_t)S * U * d.rnb_u;
  d.wg_i_elems = (size_t)S * I * d.rnb_i;
  d.partial_elems = (size_t)S * kPrSlabs * d.NA_e * R * d.NBp_e;
  d.lmax = N / MMSBM_PIECE_LEN + 1;                 // must match graph_build.cu
  d.smax = 2 * (N / MMSBM_PIECE_LEN) + 1;           // slots: at most deg/PIECE_LEN + 1 per long segment
  d.pmax_u = (int64_t)U + N / MMSBM_PIECE_LEN + 1;
  d.pmax_i = (int64_t)I + N / MMSBM_PIECE_LEN + 1;
  d.slots_u_elems = (size_t)S * d.smax * d.rnb_u;
  d.slots_i_elems = (size_t)S * d.smax * d.rnb_i;
  d.th2_elems = (size_t)(S / 2) * 2 * U * d.ldk;
  d.et2_elems = (size_t)(S / 2) * 2 * I * d.ldl;
  d.et6_elems = (size_t)(S / 6) * 6 * I * d.ldl;
  d.ctr_elems = 2 * ((size_t)S + 8);
  return d;
}

static size_t em_main_bytes(const EmDims& d) {
  return 4 * align_up(d.p_elems * 8) + align_up(d.wg_u_elems * 8) + align_up(d.wg_i_elems * 8) +
         align_up(d.partial_elems * 8) + align_up(d.slots_u_elems * 8) + align_up(d.slots_i_elems * 8) +
         align_up(d.th2_elems * 8) + align_up(d.et2_elems * 8) + align_up(d.et6_elems * 8) + align_up(d.ctr_elems * 4) + 256;
}

}  // namespace mmsbm

using namespace mmsbm;

extern "C" int mmsbm_em_workspace_bytes(int64_t N, int32_t U, int32_t I, int32_t R, int32_t K,
                                        int32_t L, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_em_workspace_bytes: bad argument");
  EmDims d = em_dims(N, U, I, R, K, L, S);
  *bytes = em_main_bytes(d);
  // the cooperative small-problem path (em_small.cu) keeps one partial n_pr per CTA behind the rest
  if (em_small_applicable(N, R, K, L, S)) *bytes += align_up(em_small_partial_elems(R, K) * 8);
  return 0;
}

// Optional second stream for the kernels that are off the critical path of an iteration
// (w of the items, both n contractions): they are HBM-streaming while the segment passes are
// bound by the L1/LSU pipe, so they overlap well.  Created per mmsbm_em_run call.
struct Overlap {
  // the caller read the two schedules: no segment is cut into pieces, the fix-up launches are skipped
  bool no_long_u = false, no_long_i = false;
  cudaStream_t side = nullptr;
  cudaEvent_t e[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  // Launch-bound sizes: the user side and the item side of an iteration only meet at the P tables,
  // so they run as two independent branches (main stream: w, by-user pass, n of the users; side
  // stream: w, by-item pass, n of the items), pr on the branch that emits it.  The critical path of
  // an iteration drops from 13 dependent kernels to 7, and the two passes fill the GPU together.
  bool two_branch = false;
};

static int em_step_impl(const int32_t* useg, const int32_t* uadj, const int32_t* udeg,
                        const int32_t* iseg, const int32_t* iadj, const int32_t* ideg,
                        const int32_t* usched, const int32_t* isched, int64_t N, int32_t U, int32_t I, int32_t R, int32_t K, int32_t L,
                        int32_t S, const double* theta, const double* eta, const double* pr,
                        double* theta_out, double* eta_out, double* pr_out, int32_t flags,
                        void* ws, size_t ws_bytes, void* stream, cudaEvent_t* ev,
                        const Overlap* ov = nullptr) {
  MMSBM_REQUIRE(useg && uadj && udeg && iseg && iadj && ideg && usched && isched && theta && eta && pr &&
                    theta_out && eta_out && pr_out && ws, MMSBM_EINVAL, "mmsbm_em_step: null pointer");
  MMSBM_REQUIRE(N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_em_step: bad size");
  MMSBM_REQUIRE(K <= 256 && L <= 256 && R <= 31, MMSBM_ERANGE,
                "mmsbm_em_step: K, L <= 256 and R <= 31 supported (K=%d L=%d R=%d)", K, L, R);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  EmDims d = em_dims(N, U, I, R, K, L, S);
  // run groups of the two segment passes: their interleaved tables are filled below
  const RunPlan plan_u = plan_runs(d.ldl, R, S, true), plan_i = plan_runs(d.ldk, R, S, false);
  Arena arena(ws, ws_bytes);
  double* pw_u = arena.take<double>(d.p_elems);
  double* pn_u = arena.take<double>(d.p_elems);
  double* pw_i = arena.take<double>(d.p_elems);
  double* pn_i = arena.take<double>(d.p_elems);
  double* wg_u = arena.take<double>(d.wg_u_elems);
  double* wg_i = arena.take<double>(d.wg_i_elems);
  double* partial = arena.take<double>(d.partial_elems);
  double* slots_u = arena.take<double>(d.slots_u_elems);
  double* slots_i = arena.take<double>(d.slots_i_elems);
  double* th2 = arena.take<double>(d.th2_elems);
  double* et2 = arena.take<double>(d.et2_elems);
  double* et6 = arena.take<double>(d.et6_elems);
  int32_t* counters = arena.take<int32_t>(d.ctr_elems);
  MMSBM_REQUIRE(pw_u && pn_u && pw_i && pn_i && wg_u && wg_i && partial && slots_u && slots_i && th2 && et2 && et6 && counters,
                MMSBM_ENOMEM,
                "mmsbm_em_step: workspace too small (%zu)", ws_bytes);
  int rc;
  // launch-wide piece queues (persistent CTAs) for large problems: immune to skewed degrees
  // (ML-20M shape with Zipf ids: 7.33 -> 5.95 ms/iteration) and to wave quantisation; small
  // problems keep per-CTA piece ranges (no counter reset, 1-6 % faster below ~1M ratings).
  // MMSBM_DYN=0/1 forces one or the other.
  const bool dyn = env_int("MMSBM_DYN", N >= ((int64_t)1 << 22) ? 1 : 0) != 0;
#define MMSBM_MARK(k) do { if (ev) MMSBM_CUDA(cudaEventRecord(ev[k], st)); } while (0)
  MMSBM_MARK(0);
  cudaStream_t s2 = ov ? ov->side : st;        // stream of the off-critical-path kernels
#define MMSBM_FORK(k) do { if (ov) { MMSBM_CUDA(cudaEventRecord(ov->e[k], st)); \
                                     MMSBM_CUDA(cudaStreamWaitEvent(s2, ov->e[k], 0)); } } while (0)
#define MMSBM_JOIN(k) do { if (ov) { MMSBM_CUDA(cudaEventRecord(ov->e[k], s2)); \
                                     MMSBM_CUDA(cudaStreamWaitEvent(st, ov->e[k], 0)); } } while (0)
#define MMSBM_SIDE_DONE(k) do { if (ov) MMSBM_CUDA(cudaEventRecord(ov->e[k], s2)); } while (0)
  if (ov && ov->two_branch) {
    if (dyn) MMSBM_CUDA(cudaMemsetAsync(counters, 0, d.ctr_elems * 4, st));
    if ((rc = launch_prep_p(pr, K, L, R, d.ldk, d.ldl, S, pw_u, pn_u, pw_i, pn_i, st))) return rc;
    MMSBM_FORK(0);
    auto pr_step = [&](cudaStream_t s) {
      return launch_pr(d.emit_items ? eta : theta, d.emit_items ? wg_i : wg_u, partial, pr, pr_out, d.nseg_e,
                       d.NA_e, d.emit_items ? d.ldl : d.ldk, d.NBp_e, K, L, R, S, d.emit_items,
                       (flags & MMSBM_RAW_ETA_PR) == 0, s);
    };
    // user branch (main stream)
    if ((rc = launch_interleave(eta, et6, I, I, 0, d.ldl, 0, plan_u.hexas, 6, st))) return rc;
    if ((rc = launch_interleave(eta, et2, I, I, 0, d.ldl, plan_u.pair_group0, plan_u.pairs, 2, st))) return rc;
    if ((rc = launch_w(theta, pw_u, wg_u, U, d.ldk, d.rnb_u, S, st))) return rc;
    {
      SegArgs a{useg, uadj, usched, eta, wg_u, slots_u, d.pmax_u, d.lmax, d.smax, U, I, d.ldl, R, 0, 0, 0,
                dyn ? counters : nullptr};
      if ((rc = launch_segment_pass_and_fixup(a, et2, et6, N, S, st, ov->no_long_u))) return rc;
    }
    if ((rc = launch_n(wg_u, pn_u, theta, udeg, theta_out, U, d.ldk, d.rnb_u,
                       (flags & MMSBM_RAW_THETA) ? 0 : 1, S, st))) return rc;
    if (!d.emit_items && (rc = pr_step(st))) return rc;
    // item branch (side stream)
    if ((rc = launch_interleave(theta, th2, U, U, 0, d.ldk, plan_i.pair_group0, plan_i.pairs, 2, s2))) return rc;
    if ((rc = launch_w(eta, pw_i, wg_i, I, d.ldl, d.rnb_i, S, s2))) return rc;
    {
      SegArgs a{iseg, iadj, isched, theta, wg_i, slots_i, d.pmax_i, d.lmax, d.smax, I, U, d.ldk, R, 0, 0, 0,
                dyn ? counters + d.ctr_elems / 2 : nullptr};
      if ((rc = launch_segment_pass_and_fixup(a, th2, nullptr, N, S, s2, ov->no_long_i))) return rc;
    }
    if ((rc = launch_n(wg_i, pn_i, eta, ideg, eta_out, I, d.ldl, d.rnb_i,
                       (flags & MMSBM_RAW_ETA_PR) ? 0 : 1, S, s2))) return rc;
    if (d.emit_items && (rc = pr_step(s2))) return rc;
    MMSBM_JOIN(1);
    return 0;
  }
  // ---- P tables and w = own x Pw for every user and item ----
  {
    if (dyn) MMSBM_CUDA(cudaMemsetAsync(counters, 0, d.ctr_elems * 4, st));   // piece queues of both passes
    if ((rc = launch_prep_p(pr, K, L, R, d.ldk, d.ldl, S, pw_u, pn_u, pw_i, pn_i, st))) return rc;
    MMSBM_FORK(0);                                                  // side: after the P tables
    // rows of run groups side by side: eta for the by-user pass (six runs when rows hold 20
    // doubles, pairs), theta for the by-item pass (pairs)
    if ((rc = launch_interleave(eta, et6, I, I, 0, d.ldl, 0, plan_u.hexas, 6, st))) return rc;
    if ((rc = launch_interleave(eta, et2, I, I, 0, d.ldl, plan_u.pair_group0, plan_u.pairs, 2, st))) return rc;
    if ((rc = launch_interleave(theta, th2, U, U, 0, d.ldk, plan_i.pair_group0, plan_i.pairs, 2, st))) return rc;
    if ((rc = launch_w(theta, pw_u, wg_u, U, d.ldk, d.rnb_u, S, st))) return rc;
    if ((rc = launch_w(eta, pw_i, wg_i, I, d.ldl, d.rnb_i, S, s2))) return rc;
    MMSBM_SIDE_DONE(1);                                             // w of the items ready
  }
  MMSBM_MARK(1);
  // ---- by-user pass: g of every user (gathers eta rows) ----
  {
    SegArgs a{useg, uadj, usched, eta, wg_u, slots_u, d.pmax_u, d.lmax, d.smax, U, I, d.ldl, R, 0, 0, 0,
              dyn ? counters : nullptr};
    if ((rc = launch_segment_pass_and_fixup(a, et2, et6, N, S, st, ov && ov->no_long_u))) return rc;
  }
  MMSBM_MARK(2);
  // theta' = (g x Pn) o theta / max(deg,1): off the critical path, overlaps the by-item pass
  MMSBM_FORK(2);
  if ((rc = launch_n(wg_u, pn_u, theta, udeg, theta_out, U, d.ldk, d.rnb_u,
                     (flags & MMSBM_RAW_THETA) ? 0 : 1, S, s2))) return rc;
  MMSBM_SIDE_DONE(4);
  MMSBM_MARK(3);
  // ---- by-item pass: g of every item (gathers theta rows) ----
  if (ov) MMSBM_CUDA(cudaStreamWaitEvent(st, ov->e[1], 0));
  {
    SegArgs a{iseg, iadj, isched, theta, wg_i, slots_i, d.pmax_i, d.lmax, d.smax, I, U, d.ldk, R, 0, 0, 0,
              dyn ? counters + d.ctr_elems / 2 : nullptr};
    // (pairs only: six interleaved theta tables of 138k users would not fit L2)
    if ((rc = launch_segment_pass_and_fixup(a, th2, nullptr, N, S, st, ov && ov->no_long_i))) return rc;
  }
  MMSBM_MARK(4);
  // eta' likewise; overlaps the pr kernels
  MMSBM_FORK(3);
  if ((rc = launch_n(wg_i, pn_i, eta, ideg, eta_out, I, d.ldl, d.rnb_i,
                     (flags & MMSBM_RAW_ETA_PR) ? 0 : 1, S, s2))) return rc;
  MMSBM_SIDE_DONE(5);
  MMSBM_MARK(5);
  // ---- pr' ----
  if ((rc = launch_pr(d.emit_items ? eta : theta, d.emit_items ? wg_i : wg_u, partial, pr, pr_out, d.nseg_e,
                      d.NA_e, d.emit_items ? d.ldl : d.ldk, d.NBp_e, K, L, R, S, d.emit_items,
                      (flags & MMSBM_RAW_ETA_PR) == 0, st))) return rc;
  MMSBM_MARK(6);
  MMSBM_MARK(7);
  if (ov) {                                                         // join: theta' and eta' are ready
    MMSBM_CUDA(cudaStreamWaitEvent(st, ov->e[4], 0));
    MMSBM_CUDA(cudaStreamWaitEvent(st, ov->e[5], 0));
  }
#undef MMSBM_MARK
#undef MMSBM_FORK
#undef MMSBM_JOIN
#undef MMSBM_SIDE_DONE
  return 0;
}

extern "C" int mmsbm_em_step(const int32_t* useg, const int32_t* uadj, const int32_t* udeg,
                             const int32_t* iseg, const int32_t* iadj, const int32_t* ideg, const int32_t* usched,
                 const int32_t* isched,
                             int64_t N, int32_t U, int32_t I, int32_t R, int32_t K, int32_t L,
                             int32_t S, const double* theta, const double* eta, const double* pr,
                             double* theta_out, double* eta_out, double* pr_out, int32_t flags,
                             void* ws, size_t ws_bytes, void* stream) {
  return em_step_impl(useg, uadj, udeg, iseg, iadj, ideg, usched, isched, N, U, I, R, K, L, S, theta, eta, pr,
                      theta_out, eta_out, pr_out, flags, ws, ws_bytes, stream, nullptr);
}

// Same step with CUDA events between its stages; synchronises the stream and writes the device
// time in ms of {P tables + w contractions, by-user pass, n contraction (users), by-item pass,
// n contraction (items), pr accumulate, pr finalize}.
extern "C" int mmsbm_em_step_profiled(const int32_t* useg, const int32_t* uadj, const int32_t* udeg,
                                      const int32_t* iseg, const int32_t* iadj, const int32_t* ideg, const int32_t* usched,
                 const int32_t* isched,
                                      int64_t N, int32_t U, int32_t I, int32_t R, int32_t K,
                                      int32_t L, int32_t S, const double* theta, const double* eta,
                                      const double* pr, double* theta_out, double* eta_out,
                                      double* pr_out, int32_t flags, void* ws, size_t ws_bytes,
                                      void* stream, float* ms7) {
  MMSBM_REQUIRE(ms7, MMSBM_EINVAL, "mmsbm_em_step_profiled: null output");
  cudaEvent_t ev[8];
  for (int k = 0; k < 8; ++k) MMSBM_CUDA(cudaEventCreate(&ev[k]));
  int rc = em_step_impl(useg, uadj, udeg, iseg, iadj, ideg, usched, isched, N, U, I, R, K, L, S, theta, eta, pr,
                        theta_out, eta_out, pr_out, flags, ws, ws_bytes, stream, ev);
  if (rc == 0) {
    cudaError_t e = cudaEventSynchronize(ev[7]);
    if (e != cudaSuccess) { set_error("cudaEventSynchronize: %s", cudaGetErrorString(e)); rc = (int)e; }
    for (int k = 0; k < 7 && rc == 0; ++k) cudaEventElapsedTime(&ms7[k], ev[k], ev[k + 1]);
  }
  for (int k = 0; k < 8; ++k) cudaEventDestroy(ev[k]);
  return rc;
}

extern "C" int mmsbm_em_run(const int32_t* useg, const int32_t* uadj, const int32_t* udeg,
                            const int32_t* iseg, const int32_t* iadj, const int32_t* ideg, const int32_t* usched,
                 const int32_t* isched,
                            int64_t N, int32_t U, int32_t I, int32_t R, int32_t K, int32_t L,
                            int32_t S, int32_t iterations, double* theta_a, double* eta_a,
                            double* pr_a, double* theta_b, double* eta_b, double* pr_b, void* ws,
                            size_t ws_bytes, void* stream) {
  MMSBM_REQUIRE(iterations >= 0, MMSBM_EINVAL, "mmsbm_em_run: negative iteration count");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // small one-run problems: the whole loop in one cooperative launch (em_small.cu)
  if (iterations > 0 && N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && em_small_applicable(N, R, K, L, S) &&
      useg && uadj && udeg && iseg && iadj && ideg && usched && isched && theta_a && eta_a && pr_a && theta_b &&
      eta_b && pr_b && ws) {
    const size_t main_bytes = em_main_bytes(em_dims(N, U, I, R, K, L, S));
    const size_t part_elems = em_small_partial_elems(R, K);
    if (ws_bytes >= main_bytes + part_elems * 8) {
      const int rc = launch_em_small(useg, uadj, udeg, iseg, iadj, ideg, usched, isched, N, U, I, R, K, L, S,
                                     iterations, theta_a, eta_a, pr_a, theta_b, eta_b, pr_b,
                                     reinterpret_cast<double*>(static_cast<char*>(ws) + main_bytes), part_elems, st);
      if (rc != MMSBM_ERANGE) return rc;
    }
  }
  Overlap ov;
  const bool small = (double)N * S < 5.0e7;
  const bool overlap = iterations > 0 && getenv("MMSBM_NO_OVERLAP") == nullptr;
  if (overlap) {
    MMSBM_CUDA(cudaStreamCreateWithFlags(&ov.side, cudaStreamNonBlocking));
    for (auto& e : ov.e) MMSBM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ov.two_branch = small && getenv("MMSBM_FORCE_OVERLAP") == nullptr;
  }
  {
    // launch-bound sizes: read the headers of the two schedules once (16 bytes each; the only host
    // synchronisation of the call) -- without long segments two launches per iteration go away
    cudaStreamCaptureStatus cs0 = cudaStreamCaptureStatusNone;
    if (small && iterations >= 8 && cudaStreamIsCapturing(st, &cs0) == cudaSuccess && cs0 == cudaStreamCaptureStatusNone) {
      int32_t hu[4] = {0, 0, 1, 0}, hi[4] = {0, 0, 1, 0};
      MMSBM_CUDA(cudaMemcpyAsync(hu, usched, sizeof(hu), cudaMemcpyDeviceToHost, st));
      MMSBM_CUDA(cudaMemcpyAsync(hi, isched, sizeof(hi), cudaMemcpyDeviceToHost, st));
      MMSBM_CUDA(cudaStreamSynchronize(st));
      ov.no_long_u = hu[2] == 0;
      ov.no_long_i = hi[2] == 0;
    }
  }
  auto step = [&](bool fwd) {
    return em_step_impl(useg, uadj, udeg, iseg, iadj, ideg, usched, isched, N, U, I, R, K, L, S,
                        fwd ? theta_a : theta_b, fwd ? eta_a : eta_b, fwd ? pr_a : pr_b,
                        fwd ? theta_b : theta_a, fwd ? eta_b : eta_a, fwd ? pr_b : pr_a, 0, ws,
                        ws_bytes, stream, nullptr, overlap ? &ov : nullptr);
  };
  struct Cleanup {                              // the side stream drains on its own; handles are
    Overlap& o;                                 // released once their work has completed
    ~Cleanup() {
      for (auto& e : o.e) if (e) cudaEventDestroy(e);
      if (o.side) cudaStreamDestroy(o.side);
    }
  } cleanup{ov};
  int done = 0;
  // Launch-bound sizes (a few 10 us of kernels per iteration): capture one a->b->a pair of
  // iterations into a CUDA graph and replay it; the graph lives only inside this call.
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (small && getenv("MMSBM_NO_GRAPH") == nullptr && iterations >= 8 && st != nullptr && cudaStreamIsCapturing(st, &cap) == cudaSuccess &&
      cap == cudaStreamCaptureStatusNone) {
    int rc = step(true);                       // first pair uncaptured: sets function attributes
    if (rc == 0) rc = step(false);
    if (rc) return rc;
    done = 2;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    const int64_t l0 = mmsbm_launch_count();
    MMSBM_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    rc = step(true);
    if (rc == 0) rc = step(false);
    cudaError_t e = cudaStreamEndCapture(st, &graph);
    const int per_pair = (int)(mmsbm_launch_count() - l0);
    count_launch(-per_pair);                   // the capture itself launched nothing
    if (rc == 0 && e == cudaSuccess && graph) e = cudaGraphInstantiate(&exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (rc) return rc;
    if (e == cudaSuccess && exec) {
      for (; done + 2 <= iterations; done += 2) {
        MMSBM_CUDA(cudaGraphLaunch(exec, st));
        count_launch(per_pair);
      }
      cudaGraphExecDestroy(exec);              // freed asynchronously once the replays finish
    } else {
      (void)cudaGetLastError();                // graph path unavailable: fall through to plain launches
    }
  }
  for (int it = done; it < iterations; ++it) {
    int rc = step((it & 1) == 0);
    if (rc) return rc;
  }
  return 0;
}

// ---- EM to convergence ----------------------------------------------------------------------
// Check j (j = 0 at the start, then after min(j*every, max_iterations) steps) evaluates l_j of
// every run (launch_loglik); converge_latch_kernel applies the rule to the runs still active and
// converge_copy_kernel snapshots the parameters of those that stop.  Latched runs keep being
// computed by the batched kernels; nothing of theirs is written again, so their results do not
// depend on the other runs.  The check index lives on the device, so one captured chunk (steps,
// l, latch, snapshot) replays unchanged.
namespace mmsbm {

struct ConvState {
  double* lik;        // [S] l of the current check
  double* prev;       // [S] l of the run's previous check
  int32_t* active;    // [S]
  int32_t* stop;      // [S] 1: the run stops at the current check
  int32_t* ctr;       // [0] index of the next check, [1] runs still active after it
};

__global__ void converge_init_kernel(ConvState c, double* trace, int32_t* iters, int32_t* conv, int S,
                                     int ntr, int max_it) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < S * ntr) trace[t] = __longlong_as_double(0x7ff8000000000000ll);   // NaN: no entry
  if (t < S) { c.active[t] = 1; iters[t] = max_it; conv[t] = 0; }
  if (t == 0) { c.ctr[0] = 0; c.ctr[1] = S; }
}

__global__ void __launch_bounds__(256) converge_latch_kernel(ConvState c, double* trace, int32_t* iters,
                                                             int32_t* conv, int S, int ntr, int every,
                                                             int max_it, double tol) {
  __shared__ int n_active;
  const int j = c.ctr[0];
  if (threadIdx.x == 0) n_active = 0;
  __syncthreads();
  int mine = 0;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    int stop = 0;
    if (c.active[s]) {
      const double l = c.lik[s];
      trace[(size_t)s * ntr + j] = l;
      if (j > 0 && fabs(l - c.prev[s]) <= tol * fabs(l)) {
        stop = 1;
        c.active[s] = 0;
        iters[s] = min(j * every, max_it);
        conv[s] = 1;
      } else {
        c.prev[s] = l;
        ++mine;
      }
    }
    c.stop[s] = stop;
  }
  atomicAdd(&n_active, mine);   // an integer count: the order of the additions does not matter
  __syncthreads();
  if (threadIdx.x == 0) { c.ctr[0] = j + 1; c.ctr[1] = n_active; }
}

// dst <- src for the runs with pick[run] != 0: theta [U][ldk], eta [I][ldl] and pr [K*L*R] of a run
struct RunCopy {
  const double* src[3];
  double* dst[3];
  size_t n[3];        // doubles per run
};
__global__ void converge_copy_kernel(const RunCopy a, const int32_t* pick) {
  const int run = blockIdx.y;
  if (!pick[run]) return;
  for (int t = 0; t < 3; ++t) {
    const double* src = a.src[t] + (size_t)run * a.n[t];
    double* dst = a.dst[t] + (size_t)run * a.n[t];
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n[t]; i += (size_t)gridDim.x * blockDim.x)
      dst[i] = src[i];
  }
}

static int launch_run_copy(const RunCopy& a, const int32_t* pick, int S, cudaStream_t st) {
  const size_t most = a.n[0] > a.n[1] ? (a.n[0] > a.n[2] ? a.n[0] : a.n[2]) : (a.n[1] > a.n[2] ? a.n[1] : a.n[2]);
  const size_t want = (most + 255) / 256, cap = (size_t)sm_count() * 4;
  converge_copy_kernel<<<dim3((unsigned)(want < cap ? want : cap), S), 256, 0, st>>>(a, pick);
  MMSBM_LAUNCH_CHECK("converge_copy_kernel");
  return 0;
}

// the EM workspace and the l workspace share one region (they are never in use at the same time)
static size_t converge_shared_bytes(int64_t N, int U, int I, int R, int K, int L, int S) {
  size_t em = 0, lk = 0;
  mmsbm_em_workspace_bytes(N, U, I, R, K, L, S, &em);
  mmsbm_loglik_workspace_bytes(N, U, I, R, K, L, S, &lk);
  return em > lk ? em : lk;
}

}  // namespace mmsbm

extern "C" int mmsbm_em_converge_workspace_bytes(int64_t N, int32_t U, int32_t I, int32_t R, int32_t K,
                                                 int32_t L, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_em_converge_workspace_bytes: bad argument");
  const size_t snap = (size_t)S * ((size_t)U * row_stride(K) + (size_t)I * row_stride(L) + (size_t)K * L * R);
  *bytes = converge_shared_bytes(N, U, I, R, K, L, S) + align_up(snap * 8) + 2 * align_up((size_t)S * 8) +
           2 * align_up((size_t)S * 4) + align_up(2 * 4) + 256;
  return 0;
}

extern "C" int mmsbm_em_run_converge(const int32_t* useg, const int32_t* uadj, const int32_t* udeg,
                                     const int32_t* iseg, const int32_t* iadj, const int32_t* ideg,
                                     const int32_t* usched, const int32_t* isched,
                                     int64_t N, int32_t U, int32_t I, int32_t R, int32_t K, int32_t L, int32_t S,
                                     int32_t max_iterations, int32_t check_every, double tol,
                                     double* theta_a, double* eta_a, double* pr_a,
                                     double* theta_b, double* eta_b, double* pr_b,
                                     double* loglik, int32_t* iterations, int32_t* converged,
                                     void* ws, size_t ws_bytes, void* stream) {
  MMSBM_REQUIRE(useg && uadj && udeg && iseg && iadj && ideg && usched && isched && theta_a && eta_a && pr_a &&
                    theta_b && eta_b && pr_b && loglik && iterations && converged && ws, MMSBM_EINVAL,
                "mmsbm_em_run_converge: null pointer");
  MMSBM_REQUIRE(N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_em_run_converge: bad size");
  MMSBM_REQUIRE(K <= 256 && L <= 256 && R <= 31, MMSBM_ERANGE,
                "mmsbm_em_run_converge: K, L <= 256 and R <= 31 supported (K=%d L=%d R=%d)", K, L, R);
  MMSBM_REQUIRE(max_iterations >= 0 && check_every >= 2 && check_every % 2 == 0, MMSBM_EINVAL,
                "mmsbm_em_run_converge: max_iterations >= 0 and an even check_every >= 2 required (%d, %d)",
                max_iterations, check_every);
  MMSBM_REQUIRE(tol >= 0.0 && tol <= 1.7976931348623157e308, MMSBM_EINVAL,
                "mmsbm_em_run_converge: tol must be finite and >= 0");
  size_t need = 0;
  mmsbm_em_converge_workspace_bytes(N, U, I, R, K, L, S, &need);
  MMSBM_REQUIRE(ws_bytes >= need, MMSBM_ENOMEM, "mmsbm_em_run_converge: workspace too small (%zu < %zu)",
                ws_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ldk = row_stride(K), ldl = row_stride(L);
  const int c = check_every, full = max_iterations / c, rem = max_iterations - full * c;
  const int checks = full + (rem > 0 ? 1 : 0), ntr = checks + 1;
  const size_t shared = converge_shared_bytes(N, U, I, R, K, L, S);
  const size_t n_th = (size_t)U * ldk, n_et = (size_t)I * ldl, n_pr = (size_t)K * L * R;
  Arena arena(static_cast<char*>(ws) + shared, ws_bytes - shared);
  double* snap = arena.take<double>((size_t)S * (n_th + n_et + n_pr));
  ConvState cs;
  cs.lik = arena.take<double>(S);
  cs.prev = arena.take<double>(S);
  cs.active = arena.take<int32_t>(S);
  cs.stop = arena.take<int32_t>(S);
  cs.ctr = arena.take<int32_t>(2);
  MMSBM_REQUIRE(snap && cs.lik && cs.prev && cs.active && cs.stop && cs.ctr, MMSBM_ENOMEM,
                "mmsbm_em_run_converge: workspace too small");
  double* snap3[3] = {snap, snap + (size_t)S * n_th, snap + (size_t)S * (n_th + n_et)};

  // launch strategy, decided once per call as in mmsbm_em_run: the schedule headers (16 bytes each)
  int32_t hu[4] = {0, 0, 1, 0}, hi[4] = {0, 0, 1, 0};
  MMSBM_CUDA(cudaMemcpyAsync(hu, usched, sizeof(hu), cudaMemcpyDeviceToHost, st));
  MMSBM_CUDA(cudaMemcpyAsync(hi, isched, sizeof(hi), cudaMemcpyDeviceToHost, st));
  MMSBM_CUDA(cudaStreamSynchronize(st));
  const bool has_long = hu[2] != 0 || hi[2] != 0;
  const size_t part_elems = em_small_partial_elems(R, K);
  const size_t main_bytes = em_main_bytes(em_dims(N, U, I, R, K, L, S));
  bool coop = checks > 0 && em_small_applicable(N, R, K, L, S) && !has_long && shared >= main_bytes + part_elems * 8;
  Overlap ov;
  const bool small = (double)N * S < 5.0e7;
  const bool overlap = checks > 0 && getenv("MMSBM_NO_OVERLAP") == nullptr;
  ov.no_long_u = hu[2] == 0;
  ov.no_long_i = hi[2] == 0;
  struct Resources {
    cudaStream_t st;
    Overlap& o;
    cudaEvent_t done[2] = {nullptr, nullptr};
    int32_t* host = nullptr;                    // pinned: the count of active runs, one slot per check in flight
    cudaGraphExec_t exec = nullptr;
    ~Resources() {
      cudaStreamSynchronize(st);                // nothing may still write to `host`
      if (exec) cudaGraphExecDestroy(exec);
      for (auto& e : done) if (e) cudaEventDestroy(e);
      if (host) cudaFreeHost(host);
      for (auto& e : o.e) if (e) cudaEventDestroy(e);
      if (o.side) cudaStreamDestroy(o.side);
    }
  } res{st, ov};
  if (overlap) {
    MMSBM_CUDA(cudaStreamCreateWithFlags(&ov.side, cudaStreamNonBlocking));
    for (auto& e : ov.e) MMSBM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ov.two_branch = small && getenv("MMSBM_FORCE_OVERLAP") == nullptr;
  }
  for (auto& e : res.done) MMSBM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  MMSBM_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&res.host), 2 * sizeof(int32_t), cudaHostAllocDefault));

  double* a3[3] = {theta_a, eta_a, pr_a};
  double* b3[3] = {theta_b, eta_b, pr_b};
  // l of the parameters in p3, then the latch and the snapshots of the runs that stop
  auto check = [&](double* const* p3) {
    int rc = launch_loglik(useg, uadj, usched, N, U, I, R, K, L, S, p3[0], p3[1], p3[2], cs.lik, ws, shared, st);
    if (rc) return rc;
    converge_latch_kernel<<<1, 256, 0, st>>>(cs, loglik, iterations, converged, S, ntr, c, max_iterations, tol);
    MMSBM_LAUNCH_CHECK("converge_latch_kernel");
    const RunCopy cp{{p3[0], p3[1], p3[2]}, {snap3[0], snap3[1], snap3[2]}, {n_th, n_et, n_pr}};
    return launch_run_copy(cp, cs.stop, S, st);
  };
  // `steps` EM steps from the _a buffers (they end in _b when `steps` is odd), then a check
  auto chunk = [&](int steps) {
    int rc = MMSBM_ERANGE;
    if (coop) {
      rc = launch_em_small(useg, uadj, udeg, iseg, iadj, ideg, usched, isched, N, U, I, R, K, L, S, steps,
                           theta_a, eta_a, pr_a, theta_b, eta_b, pr_b,
                           reinterpret_cast<double*>(static_cast<char*>(ws) + main_bytes), part_elems, st, 0);
      if (rc == MMSBM_ERANGE) coop = false;     // device or stream not served: the multi-kernel path
      else if (rc) return rc;
    }
    if (!coop) {
      for (int it = 0; it < steps; ++it) {
        const bool fwd = (it & 1) == 0;
        rc = em_step_impl(useg, uadj, udeg, iseg, iadj, ideg, usched, isched, N, U, I, R, K, L, S,
                          fwd ? theta_a : theta_b, fwd ? eta_a : eta_b, fwd ? pr_a : pr_b,
                          fwd ? theta_b : theta_a, fwd ? eta_b : eta_a, fwd ? pr_b : pr_a, 0, ws, shared,
                          stream, nullptr, overlap ? &ov : nullptr);
        if (rc) return rc;
      }
    }
    return check((steps & 1) ? b3 : a3);
  };

  {
    const int t = S * ntr;
    converge_init_kernel<<<(t + 255) / 256, 256, 0, st>>>(cs, loglik, iterations, converged, S, ntr, max_iterations);
    MMSBM_LAUNCH_CHECK("converge_init_kernel");
    if (int rc = check(a3)) return rc;          // l_0
  }
  int per_chunk = 0;
  auto enqueue = [&](int j) {                  // check j >= 1, then the count of runs still active
    int rc;
    if (res.exec && j <= full) {
      MMSBM_CUDA(cudaGraphLaunch(res.exec, st));
      count_launch(per_chunk);
    } else if ((rc = chunk(j <= full ? c : rem))) {
      return rc;
    }
    MMSBM_CUDA(cudaMemcpyAsync(res.host + (j & 1), cs.ctr + 1, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MMSBM_CUDA(cudaEventRecord(res.done[j & 1], st));
    return 0;
  };
  int enqueued = 0;
  if (checks > 0) {
    if (int rc = enqueue(1)) return rc;
    enqueued = 1;
    // launch-bound sizes: capture one chunk into a CUDA graph (the first ran uncaptured and set the
    // function attributes) and replay it for the other full chunks
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (!coop && small && full >= 3 && st != nullptr && getenv("MMSBM_NO_GRAPH") == nullptr &&
        cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone) {
      cudaGraph_t graph = nullptr;
      const int64_t l0 = mmsbm_launch_count();
      MMSBM_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      int rc = chunk(c);
      cudaError_t e = cudaStreamEndCapture(st, &graph);
      per_chunk = (int)(mmsbm_launch_count() - l0);
      count_launch(-per_chunk);                // the capture itself launched nothing
      if (rc == 0 && e == cudaSuccess && graph) e = cudaGraphInstantiate(&res.exec, graph, 0);
      if (graph) cudaGraphDestroy(graph);
      if (rc) return rc;
      if (e != cudaSuccess) {
        res.exec = nullptr;
        (void)cudaGetLastError();              // graph path unavailable: plain launches
      }
    }
  }
  // one chunk of lookahead: chunk j+1 is enqueued before the host waits for the count of check j
  for (int j = 1; j <= checks; ++j) {
    if (j < checks) {
      if (int rc = enqueue(j + 1)) return rc;
      enqueued = j + 1;
    }
    MMSBM_CUDA(cudaEventSynchronize(res.done[j & 1]));
    if (res.host[j & 1] == 0) break;
  }
  // every run's parameters into _a: the last chunk may have ended in _b, latched runs from their snapshots
  const int steps_done = enqueued <= full ? enqueued * c : max_iterations;
  if (steps_done & 1)
    for (int t = 0; t < 3; ++t) {
      const size_t n = (size_t)S * (t == 0 ? n_th : t == 1 ? n_et : n_pr);
      MMSBM_CUDA(cudaMemcpyAsync(a3[t], b3[t], n * 8, cudaMemcpyDeviceToDevice, st));
    }
  const RunCopy back{{snap3[0], snap3[1], snap3[2]}, {theta_a, eta_a, pr_a}, {n_th, n_et, n_pr}};
  if (int rc = launch_run_copy(back, converged, S, st)) return rc;
  MMSBM_CUDA(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int mmsbm_em_finalize(double* eta, const int32_t* ideg, int32_t I, int32_t L, double* pr,
                                 int32_t K, int32_t R, int32_t S, void* stream) {
  MMSBM_REQUIRE(eta && ideg && pr && I > 0 && L > 0 && K > 0 && R > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_em_finalize: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ldl = row_stride(L);
  size_t total = (size_t)S * I * ldl;
  finalize_eta_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(eta, ideg, I, ldl, L, total);
  MMSBM_LAUNCH_CHECK("finalize_eta_kernel");
  return launch_finalize_pr(pr, S * K * L, R, st);
}
