// Fold-in of ids a fitted model has not seen: EM on the rows of the new users (or items) alone,
// with the other side and pr held fixed.  For a new user u with ratings n = (u, i_n, r_n)
//
//     a_n[k]  = sum_l eta[i_n][l] P[k][l][r_n]                  (the item-side w table of em_step.cu)
//     theta'_k = theta_k * sum_n a_n[k] / max(theta . a_n, eps) / max(deg_u, 1)
//
// which is the reference's theta update (src/kernels_numpy.py:43-79 + normalize_with_d) restricted
// to u's rows; new items are the mirror case with the user-side table sum_k theta[u][k] P[k][l][r].
// With the other side fixed the segments are independent, so every iteration runs inside one
// launch without a grid barrier:
//
//   prep_p_kernel + launch_w   the per-(neighbour, level) rows a_n, W[s][other][r*ld + own]
//   fold_plan_kernel           segments too long for one CTA's shared memory, cut into pieces
//   fold_in_kernel<TPR,J>      one warp per (run, new id) segment whose rows fit a warp's slice of
//                              shared memory, then one CTA per segment that fits the whole CTA; the
//                              rows are gathered once, every iteration re-reads them from shared
//                              memory; the own row lives in registers (J doubles per lane, a group
//                              of TPR lanes holds the row, 32/TPR ratings per warp step)
//   fold_pieces_kernel +       per iteration, for the longer segments: one CTA per piece writes
//   fold_fixup_kernel          partial sums, the fix-up adds them in piece order and updates the row
//
// Every sum has a fixed order (butterfly shuffles, warps added in warp order, pieces in piece
// order): results are bit-reproducible.
#include "em_internal.cuh"

namespace mmsbm {

constexpr int kFoldWarps = 8;
constexpr int kFoldThreads = kFoldWarps * 32;
constexpr int kFoldSliceBytes = 12 * 1024;   // shared memory of one warp's rows
constexpr int kPlanThreads = 1024;

struct FoldArgs {
  const int32_t *seg, *adj, *deg;      // one-side index of the new rows (graph_build_side)
  const double* W;                     // [S][n_other][R*ld]
  double* own;                         // [S][n_new][ld], updated in place
  double* partial;                     // [S][pmax][ld]   partial sums of the pieces
  const int32_t *big, *piece_first, *piece_big, *counts;   // fold_plan_kernel
  int n_new, n_other, R, ld, cap_w, cap_c, iterations;
  int64_t pmax;
};

// rows [lo, hi) of segment a (positions in adj) -> dst[(p - lo) * ld], by `nthr` threads; the level
// of a row follows from the (id, level) buckets of seg.  256-bit read-only loads of W.
__device__ __forceinline__ void gather_rows(const FoldArgs& A, int run, int a, int lo, int hi, double* dst,
                                            int tid, int nthr) {
  const int c4 = A.ld >> 2;
  const size_t rld = (size_t)A.R * A.ld;
  const double* Wr = A.W + (size_t)run * A.n_other * rld;
  const int32_t* sg = A.seg + (size_t)a * A.R;
  for (int r = 0; r < A.R; ++r) {
    const int b0 = max(sg[r], lo), b1 = min(sg[r + 1], hi);
    const int tot = (b1 - b0) * c4;
    for (int t = tid; t < tot; t += nthr) {
      const int p = b0 + t / c4, c = t - (t / c4) * c4;
      const int o = A.adj[p];
      MMSBM_DEV_CHECK(o >= 0 && o < A.n_other);
      const double4_t v = ldg256(Wr + (size_t)o * rld + (size_t)r * A.ld + 4 * c);
      double2* d = reinterpret_cast<double2*>(dst + (size_t)(p - lo) * A.ld + 4 * c);
      d[0] = make_double2(v.x, v.y);
      d[1] = make_double2(v.z, v.w);
    }
  }
}

// g = sum over rows n of row_n / max(th . row_n, eps) for the rows gid, gid + T, ... of `rows`; a
// group of TPR lanes (t = lane in group) handles one row per step, two steps in flight.  On return
// every lane holds the sum over the warp's groups for its elements k = t + TPR*j.
template <int TPR, int J>
__device__ __forceinline__ void accum_rows(const double* rows, int nrows, int ld, const double (&th)[J],
                                           double (&g)[J], int gid, int T, int t) {
#pragma unroll
  for (int j = 0; j < J; ++j) g[j] = 0.0;
  for (int base = 0; base < nrows; base += 2 * T) {             // warp-uniform trip count
    const int n0 = base + gid, n1 = n0 + T;
    double x0[J], x1[J], d0 = 0.0, d1 = 0.0;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int k = t + TPR * j;
      x0[j] = (k < ld && n0 < nrows) ? rows[(size_t)n0 * ld + k] : 0.0;
      x1[j] = (k < ld && n1 < nrows) ? rows[(size_t)n1 * ld + k] : 0.0;
      d0 = fma(th[j], x0[j], d0);
      d1 = fma(th[j], x1[j], d1);
    }
#pragma unroll
    for (int off = TPR / 2; off > 0; off >>= 1) {
      d0 += __shfl_xor_sync(kFull, d0, off);
      d1 += __shfl_xor_sync(kFull, d1, off);
    }
    const double i0 = 1.0 / fmax(d0, kEps), i1 = 1.0 / fmax(d1, kEps);   // rows past the end: x = 0
#pragma unroll
    for (int j = 0; j < J; ++j) {
      g[j] = fma(x0[j], i0, g[j]);
      g[j] = fma(x1[j], i1, g[j]);
    }
  }
#pragma unroll
  for (int off = TPR; off < 32; off <<= 1)
#pragma unroll
    for (int j = 0; j < J; ++j) g[j] += __shfl_xor_sync(kFull, g[j], off);
}

// the whole CTA over `nrows` rows in shared memory; warp partials added in warp order (every
// thread computes the same total).  Contains two __syncthreads.
template <int TPR, int J>
__device__ __forceinline__ void cta_pass(const double* rows, int nrows, int ld, const double (&th)[J],
                                         double (&g)[J], double* red) {
  constexpr int G = 32 / TPR;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, q = lane / TPR, t = lane % TPR;
  accum_rows<TPR, J>(rows, nrows, ld, th, g, warp * G + q, kFoldWarps * G, t);
  if (q == 0)
#pragma unroll
    for (int j = 0; j < J; ++j)
      if (t + TPR * j < ld) red[warp * ld + t + TPR * j] = g[j];
  __syncthreads();
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int k = t + TPR * j;
    double s = 0.0;
    if (k < ld)
      for (int w = 0; w < kFoldWarps; ++w) s += red[w * ld + k];
    g[j] = s;
  }
  __syncthreads();
}

template <int TPR, int J>
__device__ __forceinline__ void load_row(const double* p, int ld, double (&th)[J], int t) {
#pragma unroll
  for (int j = 0; j < J; ++j) th[j] = (t + TPR * j < ld) ? p[t + TPR * j] : 0.0;
}

template <int TPR, int J>
__device__ __forceinline__ void store_row(double* p, int ld, const double (&th)[J], int t) {
#pragma unroll
  for (int j = 0; j < J; ++j)
    if (t + TPR * j < ld) p[t + TPR * j] = th[j];
}

// CTA b serves the new ids [8b, 8b+8) of run blockIdx.y: first one warp per id with at most cap_w
// rows, then the whole CTA for each id with cap_w < deg <= cap_c, in id order.
template <int TPR, int J>
__global__ void __launch_bounds__(kFoldThreads) fold_in_kernel(const FoldArgs A) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  double* rows = reinterpret_cast<double*>(smem_raw);            // [cap_c][ld] = [8][cap_w][ld]
  double* red = rows + (size_t)A.cap_c * A.ld;                    // [8][ld]
  constexpr int G = 32 / TPR;
  const int run = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane / TPR, t = lane % TPR;
  const int a0 = blockIdx.x * kFoldWarps;
  double* own_run = A.own + (size_t)run * A.n_new * A.ld;
  double th[J], g[J];
  {
    const int a = a0 + warp;
    const int deg = a < A.n_new ? A.deg[a] : A.cap_w + 1;
    if (deg <= A.cap_w) {
      const int lo = A.seg[(size_t)a * A.R];
      double* mine = rows + (size_t)warp * A.cap_w * A.ld;
      gather_rows(A, run, a, lo, lo + deg, mine, lane, 32);
      __syncwarp();
      load_row<TPR, J>(own_run + (size_t)a * A.ld, A.ld, th, t);
      const double dd = (double)max(deg, 1);
      for (int it = 0; it < A.iterations; ++it) {
        accum_rows<TPR, J>(mine, deg, A.ld, th, g, q, G, t);
#pragma unroll
        for (int j = 0; j < J; ++j) th[j] = th[j] * g[j] / dd;
      }
      if (q == 0) store_row<TPR, J>(own_run + (size_t)a * A.ld, A.ld, th, t);
    }
  }
  const int a1 = min(a0 + kFoldWarps, A.n_new);
  for (int a = a0; a < a1; ++a) {
    const int deg = A.deg[a];
    if (deg <= A.cap_w || deg > A.cap_c) continue;               // CTA-uniform
    __syncthreads();                                             // shared memory free again
    const int lo = A.seg[(size_t)a * A.R];
    gather_rows(A, run, a, lo, lo + deg, rows, threadIdx.x, kFoldThreads);
    __syncthreads();
    load_row<TPR, J>(own_run + (size_t)a * A.ld, A.ld, th, t);
    const double dd = (double)deg;
    for (int it = 0; it < A.iterations; ++it) {
      cta_pass<TPR, J>(rows, deg, A.ld, th, g, red);
#pragma unroll
      for (int j = 0; j < J; ++j) th[j] = th[j] * g[j] / dd;
    }
    if (warp == 0 && q == 0) store_row<TPR, J>(own_run + (size_t)a * A.ld, A.ld, th, t);
  }
}

// One iteration of the segments longer than cap_c: CTAs walk the pieces (cap_c rows each) and write
// the partial sum of each; fold_fixup_kernel then updates the rows.
template <int TPR, int J>
__global__ void __launch_bounds__(kFoldThreads) fold_pieces_kernel(const FoldArgs A) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  double* rows = reinterpret_cast<double*>(smem_raw);
  double* red = rows + (size_t)A.cap_c * A.ld;
  const int run = blockIdx.y, t = (threadIdx.x & 31) % TPR;
  const int n_pieces = A.counts[1];
  const double* own_run = A.own + (size_t)run * A.n_new * A.ld;
  double th[J], g[J];
  for (int p = blockIdx.x; p < n_pieces; p += gridDim.x) {
    const int b = A.piece_big[p], a = A.big[b];
    const int start = A.seg[(size_t)a * A.R];
    const int lo = start + (p - A.piece_first[b]) * A.cap_c, hi = min(lo + A.cap_c, start + A.deg[a]);
    __syncthreads();
    gather_rows(A, run, a, lo, hi, rows, threadIdx.x, kFoldThreads);
    __syncthreads();
    load_row<TPR, J>(own_run + (size_t)a * A.ld, A.ld, th, t);
    cta_pass<TPR, J>(rows, hi - lo, A.ld, th, g, red);
    if (threadIdx.x < TPR) store_row<TPR, J>(A.partial + ((size_t)run * A.pmax + p) * A.ld, A.ld, g, t);
  }
}

__global__ void fold_fixup_kernel(const FoldArgs A) {
  const int run = blockIdx.y;
  const int n_big = A.counts[0];
  for (int b = blockIdx.x; b < n_big; b += gridDim.x) {
    const int a = A.big[b], p0 = A.piece_first[b], p1 = A.piece_first[b + 1];
    const double dd = (double)A.deg[a];
    double* row = A.own + ((size_t)run * A.n_new + a) * A.ld;
    for (int k = threadIdx.x; k < A.ld; k += blockDim.x) {
      double s = 0.0;
      for (int p = p0; p < p1; ++p) s += A.partial[((size_t)run * A.pmax + p) * A.ld + k];
      row[k] = row[k] * s / dd;
    }
  }
}

// One CTA: the segments with more than `cap` rows in id order (big), the first piece of each
// (piece_first, with a sentinel) and the segment of each piece (piece_big); counts = {big, pieces}.
__global__ void __launch_bounds__(kPlanThreads) fold_plan_kernel(const int32_t* deg, int n, int cap,
                                                                 int32_t* big, int32_t* piece_first,
                                                                 int32_t* piece_big, int32_t* counts) {
  __shared__ long long wsum[kPlanThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long off = 0;                                  // (segments << 32) | pieces before this chunk
  for (int base = 0; base < n; base += kPlanThreads) {
    const int a = base + threadIdx.x;
    const int d = a < n ? deg[a] : 0;
    const int np = d > cap ? (d + cap - 1) / cap : 0;
    const long long mine = np ? ((1ll << 32) | np) : 0;
    long long v = mine;                               // inclusive warp scan
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(kFull, v, o);
      if (lane >= o) v += u;
    }
    if (lane == 31) wsum[warp] = v;
    __syncthreads();
    if (warp == 0) {
      long long w = wsum[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(kFull, w, o);
        if (lane >= o) w += u;
      }
      wsum[lane] = w;                                 // inclusive over warps
    }
    __syncthreads();
    const long long excl = off + (warp ? wsum[warp - 1] : 0) + v - mine;
    if (np) {
      const int bi = (int)(excl >> 32), pf = (int)(excl & 0xffffffffll);
      big[bi] = a;
      piece_first[bi] = pf;
      for (int p = 0; p < np; ++p) piece_big[pf + p] = bi;
    }
    off += wsum[kPlanThreads / 32 - 1];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int nb = (int)(off >> 32), npc = (int)(off & 0xffffffffll);
    counts[0] = nb;
    counts[1] = npc;
    piece_first[nb] = npc;
  }
}

struct FoldDims {
  int ld, ld_other, cap_w, cap_c;
  int64_t nbig_max, pmax;
  size_t smem, p_elems, w_elems, partial_elems;
};

static FoldDims fold_dims(int64_t N, int side, int n_other, int R, int K, int L, int S) {
  FoldDims d;
  d.ld = row_stride(side == 0 ? K : L);
  d.ld_other = row_stride(side == 0 ? L : K);
  d.cap_w = kFoldSliceBytes / (d.ld * 8);
  d.cap_c = kFoldWarps * d.cap_w;
  d.nbig_max = N / (d.cap_c + 1) + 1;
  d.pmax = N / d.cap_c + d.nbig_max + 1;
  d.smem = ((size_t)d.cap_c + kFoldWarps) * d.ld * 8;
  d.p_elems = (size_t)S * row_stride(K) * row_stride(L) * R;
  d.w_elems = (size_t)S * n_other * R * d.ld;
  d.partial_elems = (size_t)S * d.pmax * d.ld;
  return d;
}

static size_t fold_bytes(const FoldDims& d) {
  return 4 * align_up(d.p_elems * 8) + align_up(d.w_elems * 8) + align_up(d.partial_elems * 8) +
         2 * align_up((size_t)(d.nbig_max + 1) * 4) + align_up((size_t)d.pmax * 4) + align_up(2 * 4) + 256;
}

template <int TPR, int J>
static int launch_fold(const FoldArgs& A, const FoldDims& d, int64_t N, int S, cudaStream_t st) {
  auto main_k = fold_in_kernel<TPR, J>;
  auto piece_k = fold_pieces_kernel<TPR, J>;
  MMSBM_CUDA(cudaFuncSetAttribute(main_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d.smem));
  MMSBM_CUDA(cudaFuncSetAttribute(piece_k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)d.smem));
  main_k<<<dim3((A.n_new + kFoldWarps - 1) / kFoldWarps, S), kFoldThreads, d.smem, st>>>(A);
  MMSBM_LAUNCH_CHECK("fold_in_kernel");
  if (N <= A.cap_c) return 0;            // no segment can be longer than all the rows together
  const unsigned gp = (unsigned)(d.pmax < sm_count() * 2 ? d.pmax : sm_count() * 2);
  const unsigned gb = (unsigned)(d.nbig_max < sm_count() * 4 ? d.nbig_max : sm_count() * 4);
  for (int it = 0; it < A.iterations; ++it) {
    piece_k<<<dim3(gp, S), kFoldThreads, d.smem, st>>>(A);
    MMSBM_LAUNCH_CHECK("fold_pieces_kernel");
    fold_fixup_kernel<<<dim3(gb, S), 128, 0, st>>>(A);
    MMSBM_LAUNCH_CHECK("fold_fixup_kernel");
  }
  return 0;
}

}  // namespace mmsbm

using namespace mmsbm;

extern "C" int mmsbm_fold_in_workspace_bytes(int64_t n_ratings, int32_t side, int32_t n_new, int32_t n_other,
                                             int32_t R, int32_t K, int32_t L, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && n_ratings >= 0 && (side == 0 || side == 1) && n_new > 0 && n_other > 0 && R > 0 &&
                    K > 0 && L > 0 && S > 0, MMSBM_EINVAL, "mmsbm_fold_in_workspace_bytes: bad argument");
  *bytes = fold_bytes(fold_dims(n_ratings, side, n_other, R, K, L, S));
  return 0;
}

extern "C" int mmsbm_fold_in(const int32_t* seg, const int32_t* adj, const int32_t* deg, int64_t n_ratings,
                             int32_t side, int32_t n_new, int32_t n_other, int32_t R, int32_t K, int32_t L,
                             int32_t S, int32_t iterations, const double* other, const double* pr, double* own,
                             void* ws, size_t ws_bytes, void* stream) {
  MMSBM_REQUIRE(seg && deg && other && pr && own && ws && (n_ratings == 0 || adj), MMSBM_EINVAL,
                "mmsbm_fold_in: null pointer");
  MMSBM_REQUIRE(n_ratings >= 0 && (side == 0 || side == 1) && n_new > 0 && n_other > 0 && R > 0 && K > 0 &&
                    L > 0 && S > 0 && S <= 65535 && iterations >= 0, MMSBM_EINVAL, "mmsbm_fold_in: bad size");
  MMSBM_REQUIRE(K <= 256 && L <= 256 && R <= 31 && n_ratings < ((int64_t)1 << 31) &&
                    (int64_t)n_new * R < ((int64_t)1 << 31), MMSBM_ERANGE,
                "mmsbm_fold_in: K, L <= 256, R <= 31 and n_ratings, n_new*R < 2^31 supported "
                "(K=%d L=%d R=%d)", K, L, R);
  if (iterations == 0) return 0;
  const FoldDims d = fold_dims(n_ratings, side, n_other, R, K, L, S);
  MMSBM_REQUIRE(ws_bytes >= fold_bytes(d), MMSBM_ENOMEM, "mmsbm_fold_in: workspace %zu < %zu", ws_bytes,
                fold_bytes(d));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Arena arena(ws, ws_bytes);
  double* pw_u = arena.take<double>(d.p_elems);
  double* pn_u = arena.take<double>(d.p_elems);
  double* pw_i = arena.take<double>(d.p_elems);
  double* pn_i = arena.take<double>(d.p_elems);
  double* W = arena.take<double>(d.w_elems);
  double* partial = arena.take<double>(d.partial_elems);
  int32_t* big = arena.take<int32_t>(d.nbig_max + 1);
  int32_t* piece_first = arena.take<int32_t>(d.nbig_max + 1);
  int32_t* piece_big = arena.take<int32_t>(d.pmax);
  int32_t* counts = arena.take<int32_t>(2);
  MMSBM_REQUIRE(counts, MMSBM_ENOMEM, "mmsbm_fold_in: workspace carve-up failed");
  int rc;
  const int ldk = row_stride(K), ldl = row_stride(L);
  if ((rc = launch_prep_p(pr, K, L, R, ldk, ldl, S, pw_u, pn_u, pw_i, pn_i, st))) return rc;
  // a_n rows: new users read the item-side table (eta x Pw_i), new items the user-side one
  if ((rc = launch_w(other, side == 0 ? pw_i : pw_u, W, n_other, d.ld_other, R * d.ld, S, st))) return rc;
  fold_plan_kernel<<<1, kPlanThreads, 0, st>>>(deg, n_new, d.cap_c, big, piece_first, piece_big, counts);
  MMSBM_LAUNCH_CHECK("fold_plan_kernel");
  FoldArgs A{seg, adj, deg, W, own, partial, big, piece_first, piece_big, counts,
             n_new, n_other, R, d.ld, d.cap_w, d.cap_c, iterations, d.pmax};
  switch (d.ld) {
    case 4: return launch_fold<4, 1>(A, d, n_ratings, S, st);
    case 8: return launch_fold<8, 1>(A, d, n_ratings, S, st);
    case 12: case 16: return launch_fold<8, 2>(A, d, n_ratings, S, st);
    case 20: case 24: return launch_fold<8, 3>(A, d, n_ratings, S, st);
    case 28: case 32: return launch_fold<8, 4>(A, d, n_ratings, S, st);
    default: break;
  }
  switch ((d.ld + 31) / 32) {
    case 2: return launch_fold<32, 2>(A, d, n_ratings, S, st);
    case 3: return launch_fold<32, 3>(A, d, n_ratings, S, st);
    case 4: return launch_fold<32, 4>(A, d, n_ratings, S, st);
    case 5: return launch_fold<32, 5>(A, d, n_ratings, S, st);
    case 6: return launch_fold<32, 6>(A, d, n_ratings, S, st);
    case 7: return launch_fold<32, 7>(A, d, n_ratings, S, st);
    default: return launch_fold<32, 8>(A, d, n_ratings, S, st);
  }
}
