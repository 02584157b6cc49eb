// On-device reductions around the EM loop: the reference's "likelihood"
// (src/expectation_maximization.py:157-167), prod_dist (src/kernels_numpy.py:86-97), the
// prediction statistics (src/mmsbm.py:488-539), the mean over runs (src/mmsbm.py:315) and a
// materialising compute_omegas (src/kernels_numpy.py:21-36) for the plugin shim.
// All sums are two-stage with a fixed order (bit-reproducible).
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "em_internal.cuh"    // sm_count()
#include "segment_pass.cuh"   // double4_t, ldg256, GroupSum (lane groups of the row gathers)

namespace mmsbm {

constexpr int kLikWarps = 8;
constexpr int kLikCtas = 148 * 4;   // CTAs per run of the element-wise kernel (sizes its partial-sum buffer; a B200 has 148 SMs)

// ---- likelihood ----------------------------------------------------------------------------
// sum_n sum_kl w~ (log w~ - log S~_n), w~ = max(theta_k eta_l pr_klr, eps), S~ = max(sum w, eps).
// The clamp acts on each (k,l), so every rating costs K*L element visits; what can be saved is
// the logarithm: for w >= eps, log w = log theta_k + log eta_l + log pr_klr (three table values,
// exact to rounding), for w < eps it is the constant log eps.  One log per (rating, l) remains.
// Per rating: sum_kl w~ log w~ - log S~ * sum_kl w~, in a single sweep over k.
// One warp walks whole user segments of the (user, level)-grouped index: theta_u and its logs
// are staged once per user, the level is implied by the group; lanes own l, the loop runs over k.
struct LikArgs {
  const int32_t* useg; const int32_t* uadj;
  const double* theta; const double* eta; const double* pr;
  double* partial;      // [S][kLikCtas*kLikWarps]
  double* tables;       // [S][2][R][K][L] in global memory when they do not fit shared memory
  int U, I, R, K, L, ldk, ldl;
  const int* redo;      // [S] or null: only the runs with redo[run] != 0 are evaluated
};

// pr and log pr in [R][K][L] order (global-memory variant of the tables)
__global__ void lik_tables_kernel(const double* pr, int K, int L, int R, double* tables, const int* redo) {
  const int run = blockIdx.y, n = K * L * R;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n || (redo && !redo[run])) return;
  const int kl = t / R, r = t - kl * R;
  const double v = __ldg(pr + (size_t)run * n + t);
  double* base = tables + (size_t)run * 2 * n;
  base[(size_t)r * K * L + kl] = v;
  base[(size_t)n + (size_t)r * K * L + kl] = log(v);
}

__global__ void __launch_bounds__(kLikWarps * 32) likelihood_kernel(const LikArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = A.K, L = A.L, R = A.R;
  const double kLogEps = log(kEps);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int run = blockIdx.y;
  if (A.redo && !A.redo[run]) return;                        // the factorised total of this run stands
  const double* Pq;                                          // [R][K][L]
  const double* Lq;                                          // [R][K][L]  log pr
  double* th_s;                                              // [warps][2][K]  theta, log theta
  if (A.tables) {                                            // tables too large for shared memory
    Pq = A.tables + (size_t)run * 2 * K * L * R;
    Lq = Pq + (size_t)K * L * R;
    th_s = reinterpret_cast<double*>(smem_raw);
  } else {
    double* Ps = reinterpret_cast<double*>(smem_raw);
    double* Ls = Ps + (size_t)R * K * L;
    th_s = Ls + (size_t)R * K * L;
    const double* prs = A.pr + (size_t)run * K * L * R;
    for (int t = threadIdx.x; t < K * L * R; t += blockDim.x) {
      int kl = t / R, r = t - kl * R;
      const double v = __ldg(prs + t);
      Ps[(size_t)r * K * L + kl] = v;
      Ls[(size_t)r * K * L + kl] = log(v);
    }
    __syncthreads();
    Pq = Ps; Lq = Ls;
  }
  double* th = th_s + warp * 2 * K;
  double* lth = th + K;
  const double* theta_run = A.theta + (size_t)run * A.U * A.ldk;
  const double* eta_run = A.eta + (size_t)run * A.I * A.ldl;
  const int gw = blockIdx.x * kLikWarps + warp, nw = gridDim.x * kLikWarps;
  double acc = 0.0;
  for (int u = gw; u < A.U; u += nw) {
    __syncwarp();
    for (int k = lane; k < K; k += 32) {
      const double v = __ldg(theta_run + (size_t)u * A.ldk + k);
      th[k] = v;
      lth[k] = log(v);
    }
    __syncwarp();
    for (int r = 0; r < R; ++r) {
      const int lo = __ldg(A.useg + (size_t)u * R + r), hi = __ldg(A.useg + (size_t)u * R + r + 1);
      const double* Pr = Pq + (size_t)r * K * L;
      const double* Lr = Lq + (size_t)r * K * L;
      for (int j = lo; j < hi; ++j) {
        const int item = __ldg(A.uadj + j);
        MMSBM_DEV_CHECK(item >= 0 && item < A.I);
        const double* erow = eta_run + (size_t)item * A.ldl;
        double tot = 0.0, s1 = 0.0, s2 = 0.0;   // sum w, sum w~ log w~, sum w~
        for (int l0 = 0; l0 < L; l0 += 32) {
          const int l = l0 + lane;
          if (l < L) {
            const double e = __ldg(erow + l);
            const double le = log(e);
            for (int k = 0; k < K; ++k) {
              const double w = __dmul_rn(__dmul_rn(th[k], e), Pr[k * L + l]);   // reference order
              const bool small = w < kEps;
              const double wc = small ? kEps : w;
              const double lw = small ? kLogEps : (lth[k] + le) + Lr[k * L + l];
              tot += w;
              s1 = fma(wc, lw, s1);
              s2 += wc;
            }
          }
        }
        tot = warp_sum(tot);
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        acc += s1 - log(fmax(tot, kEps)) * s2;
      }
    }
  }
  if (lane == 0) A.partial[(size_t)run * nw + gw] = acc;
}

// ---- likelihood, factorised ---------------------------------------------------------------
// For elements that are not clamped, sum_kl w log w splits into the same bilinear forms as the EM
// step (w = theta_k eta_l p_klr, so log w = log theta_k + log eta_l + log p_klr):
//     S_n = <W_{u,r}, eta_i>                       W[l] = sum_k theta_k p_klr
//     T_n = <A_{u,r}, eta_i> + <W_{u,r}, eta_i log eta_i>
//                                                  A[l] = sum_k (theta_k log theta_k) p_klr + theta_k (p log p)_klr
//     likelihood = sum_n T_n - S_n log max(S_n, eps)
// i.e. O(K+L) per rating after two per-(user, level) tables, instead of K*L element visits and
// L logarithms.  x log x := 0 at x = 0.  The reference clamps every w below eps up to eps
// (src/expectation_maximization.py:162-166); here such an element contributes w (log w - log S~)
// instead of eps (log eps - log S~), a difference of at most eps (2 |log eps| + |log S~_n|).  Over
// a run that is at most K L eps (2 N |log eps| + sum_n |log S~_n|), which the pass bounds by also
// summing |log S~_n|.  On dense parameters the bound is ~1e-12 relative to the total; on a
// converged fit with one-hot memberships the total itself shrinks toward 0 and is made of clamp
// terms, and the factorised form can be off by 100 %.  So a run whose bound exceeds 1e-9 of its
// factorised total is evaluated again by likelihood_kernel (decided on the device, lik_check_kernel).
// Walks the (user, level)-grouped index with the piece schedule of the EM step, so a heavy user
// costs no more than 2048 ratings per warp; one partial per piece, summed in piece order.
__device__ __forceinline__ double xlogx(double x) { return x > 0.0 ? x * log(x) : 0.0; }

// E2[run][item][0][:] = eta, [1][:] = eta log eta  (one contiguous 2*8*ldl-byte gather per rating)
__global__ void lik_eta_table_kernel(const double* __restrict__ eta, double* __restrict__ e2, size_t rows, int ld) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * ld) return;
  const size_t row = t / ld;
  const int c = (int)(t - row * ld);
  const double v = __ldg(eta + t);
  e2[(row * 2) * ld + c] = v;
  e2[(row * 2 + 1) * ld + c] = xlogx(v);
}

// W and A rows of every user: a lane owns a user, the two operand tables sit in shared memory
// (every read a warp broadcast).  Pw[a][o] = p, Pl[a][o] = p log p with o = r*ldl + l, zero padded.
template <int LD>
__global__ void __launch_bounds__(256) lik_user_tables_kernel(const double* __restrict__ theta,
                                                              const double* __restrict__ pr,
                                                              double* __restrict__ W, double* __restrict__ A,
                                                              int U, int K, int L, int R, int ldl, int run0) {
  extern __shared__ __align__(32) unsigned char smem_raw[];
  const int RNB = R * ldl;
  double* Pw = reinterpret_cast<double*>(smem_raw);          // [LD][RNB]
  double* Pl = Pw + (size_t)LD * RNB;
  const int run = run0 + blockIdx.y;
  const double* prs = pr + (size_t)run * K * L * R;
  for (int t = threadIdx.x; t < LD * RNB; t += blockDim.x) {
    const int a = t / RNB, o = t - a * RNB, r = o / ldl, l = o - r * ldl;
    const double v = (a < K && l < L) ? __ldg(prs + ((size_t)a * L + l) * R + r) : 0.0;
    Pw[t] = v;
    Pl[t] = xlogx(v);
  }
  __syncthreads();
  const double* th_run = theta + (size_t)run * U * LD;
  double* w_run = W + (size_t)blockIdx.y * U * RNB;
  double* a_run = A + (size_t)blockIdx.y * U * RNB;
  for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < U; m += gridDim.x * blockDim.x) {
    double o[LD], ol[LD];
#pragma unroll
    for (int c = 0; c < LD / 4; ++c) {
      const double4_t v = ldg256(th_run + (size_t)m * LD + 4 * c);
      o[4 * c] = v.x; o[4 * c + 1] = v.y; o[4 * c + 2] = v.z; o[4 * c + 3] = v.w;
    }
#pragma unroll
    for (int a = 0; a < LD; ++a) ol[a] = xlogx(o[a]);
    for (int ob = 0; ob < RNB; ob += 4) {
      double4_t w{0.0, 0.0, 0.0, 0.0}, q{0.0, 0.0, 0.0, 0.0};
#pragma unroll
      for (int a = 0; a < LD; ++a) {
        const double4_t p = lds32(Pw + a * RNB + ob);
        const double4_t pl = lds32(Pl + a * RNB + ob);
        w.x = fma(o[a], p.x, w.x); w.y = fma(o[a], p.y, w.y); w.z = fma(o[a], p.z, w.z); w.w = fma(o[a], p.w, w.w);
        q.x = fma(ol[a], p.x, q.x); q.y = fma(ol[a], p.y, q.y); q.z = fma(ol[a], p.z, q.z); q.w = fma(ol[a], p.w, q.w);
        q.x = fma(o[a], pl.x, q.x); q.y = fma(o[a], pl.y, q.y); q.z = fma(o[a], pl.z, q.z); q.w = fma(o[a], pl.w, q.w);
      }
      stg256(w_run + (size_t)m * RNB + ob, w);
      stg256(a_run + (size_t)m * RNB + ob, q);
    }
  }
}

struct LikPassArgs {
  const int32_t* useg; const int32_t* uadj; const int32_t* sched;
  const double* e2;       // [runs][I][2][NBp]; OBS: eta [runs][I][ld]
  const double* W;        // [runs][U][R*NBp]; OBS: [runs][U][R*ld]
  const double* A;        // (not read by OBS)
  double* partial;        // [runs][pmax]
  int64_t pmax;
  int U, I, R;
  int ld;                 // OBS: row stride of eta (NBp when G < 8, any multiple of 4 >= 32 when G == 8)
  double* lpartial;       // [runs][pmax] sum_n |log S~_n| of the piece (not written by OBS)
};

// One warp per piece; groups of G lanes own a rating (lane q holds doubles 4q..4q+3 of both rows).
// OBS: the observed-data log-likelihood sum_n log max(S_n, eps) instead: only W and eta rows are
// read (half the bytes per rating), and rows wider than 32 doubles are walked in slices of 32
// (lane q of the 8-lane group holds doubles 32c+4q..32c+4q+3 of slice c).
// One body, two kernels (lik_pass_kernel, loglik_pass_kernel), so each form keeps its own name.
template <int G, bool OBS>
__device__ __forceinline__ void lik_pass_body(const LikPassArgs& P) {
  constexpr int RPS = 32 / G, UN = (G == 1) ? 1 : 2, SLOTS = UN * RPS, NBp = 4 * G;
  static_assert(SLOTS <= 32, "a chunk's ids must fit one 32-lane load");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int grp = lane / G, q = lane - grp * G;
  const bool lane_on = grp < RPS;
  const int qoff = lane_on ? 4 * q : 0;
  const int LD = OBS ? P.ld : NBp, nsl = (LD + NBp - 1) / NBp;
  const int run = blockIdx.y, R = P.R, RNB = R * LD;
  const GroupSum<G> group_sum(grp * G, q);
  const int32_t* piece_seg = P.sched + 4;
  const int32_t* piece_idx = piece_seg + P.pmax;
  const int n_pieces = __ldg(P.sched);
  const double* e2 = P.e2 + (size_t)run * P.I * (OBS ? 1 : 2) * LD;
  for (int p = blockIdx.x * (blockDim.x >> 5) + warp; p < n_pieces; p += gridDim.x * (blockDim.x >> 5)) {
    const int sg = __ldg(piece_seg + p), pidx = __ldg(piece_idx + p);
    MMSBM_DEV_CHECK(sg >= 0 && sg < P.U);
    int bend = 0;
    if (lane <= R) bend = __ldg(P.useg + (size_t)sg * R + lane);
    const int beg = __shfl_sync(kFull, bend, 0) + pidx * MMSBM_PIECE_LEN;
    const int end = min(beg + MMSBM_PIECE_LEN, __shfl_sync(kFull, bend, R));
    const double* wrow = P.W + ((size_t)run * P.U + sg) * RNB;
    const double* arow = P.A + ((size_t)run * P.U + sg) * RNB;
    double acc = 0.0, lacc = 0.0;
    int lo = beg;
    for (int r = 0; r < R; ++r) {
      const int le = min(end, __shfl_sync(kFull, bend, r + 1));
      if (lo >= le) continue;
      const double* wr_row = wrow + r * LD;
      const double4_t wr = ldg256(wr_row + qoff);
      double4_t ar{0.0, 0.0, 0.0, 0.0};
      if constexpr (!OBS) ar = ldg256(arow + r * NBp + qoff);
      for (int base = lo; base < le; base += SLOTS) {
        const int cnt = min(SLOTS, le - base);
        int ids = 0;
        if (lane < cnt) ids = __ldg(P.uadj + base + lane);
        if constexpr (OBS) {
          int id[UN];
          double4_t e[UN];
          double sv[UN];
#pragma unroll
          for (int un = 0; un < UN; ++un) {
            const int sl = un * RPS + grp;
            id[un] = __shfl_sync(kFull, ids, sl & 31);
            if (sl >= cnt) id[un] = 0;
            MMSBM_DEV_CHECK(id[un] >= 0 && id[un] < P.I);
            e[un] = ldg256(e2 + (size_t)id[un] * LD + qoff);
          }
#pragma unroll
          for (int un = 0; un < UN; ++un) {
            double s = fma(e[un].x, wr.x, fma(e[un].y, wr.y, fma(e[un].z, wr.z, e[un].w * wr.w)));
            if constexpr (G == 8) {                          // rows wider than 32 doubles
              for (int c = 1; c < nsl; ++c) {
                const int off = c * NBp + qoff;
                if (off < LD) {
                  const double4_t ec = ldg256(e2 + (size_t)id[un] * LD + off), wc = ldg256(wr_row + off);
                  s = fma(ec.x, wc.x, fma(ec.y, wc.y, fma(ec.z, wc.z, fma(ec.w, wc.w, s))));
                }
              }
            }
            sv[un] = group_sum(s);
          }
#pragma unroll
          for (int un = 0; un < UN; ++un)
            if (lane_on && q == 0 && un * RPS + grp < cnt) acc += log(fmax(sv[un], kEps));
          continue;
        }
        double4_t e[UN], el[UN];
#pragma unroll
        for (int un = 0; un < UN; ++un) {
          const int sl = un * RPS + grp;
          int id = __shfl_sync(kFull, ids, sl & 31);
          if (sl >= cnt) id = 0;
          MMSBM_DEV_CHECK(id >= 0 && id < P.I);
          const double* row = e2 + (size_t)id * 2 * NBp + qoff;
          e[un] = ldg256(row);
          el[un] = ldg256(row + NBp);
        }
#pragma unroll
        for (int un = 0; un < UN; ++un) {
          double s = fma(e[un].x, wr.x, fma(e[un].y, wr.y, fma(e[un].z, wr.z, e[un].w * wr.w)));
          double t = fma(e[un].x, ar.x, fma(e[un].y, ar.y, fma(e[un].z, ar.z, e[un].w * ar.w)));
          t = fma(el[un].x, wr.x, fma(el[un].y, wr.y, fma(el[un].z, wr.z, fma(el[un].w, wr.w, t))));
          s = group_sum(s);
          t = group_sum(t);
          if (lane_on && q == 0 && un * RPS + grp < cnt) {
            const double ls = log(fmax(s, kEps));
            acc += t - s * ls;
            lacc += fabs(ls);
          }
        }
      }
      lo = le;
    }
    acc = warp_sum(acc);
    if (lane == 0) P.partial[(size_t)run * P.pmax + p] = acc;
    if constexpr (!OBS) {
      lacc = warp_sum(lacc);
      if (lane == 0) P.lpartial[(size_t)run * P.pmax + p] = lacc;
    }
  }
}

template <int G>
__global__ void __launch_bounds__(256) lik_pass_kernel(const LikPassArgs P) { lik_pass_body<G, false>(P); }

template <int G>
__global__ void __launch_bounds__(256) loglik_pass_kernel(const LikPassArgs P) { lik_pass_body<G, true>(P); }

// out[run] = the fixed-order sum of the run's n partials (only the runs with only[run] != 0 when
// only is given)
__global__ void __launch_bounds__(256) sum_partials_kernel(const double* partial, int n, double* out,
                                                           const int* only = nullptr) {
  if (only && !only[blockIdx.x]) return;
  __shared__ double sm[256];
  const double* p = partial + (size_t)blockIdx.x * n;
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) acc += p[i];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sm[0];
}

// redo[run] = 1 when what the clamps the factorised form drops could move the run's total by more
// than 1e-9 of it: K L eps (2 N |log eps| + sum_n |log S~_n|) > 1e-9 |total| (NaN totals included)
__global__ void lik_check_kernel(const double* total, const double* labs, int S, double kl_eps,
                                 double two_n_logeps, int* redo) {
  const int run = blockIdx.x * blockDim.x + threadIdx.x;
  if (run >= S) return;
  const double bound = kl_eps * (two_n_logeps + labs[run]);
  redo[run] = !(bound <= 1e-9 * fabs(total[run]));
}

// ---- prod_dist -----------------------------------------------------------------------------
struct ProdArgs {
  const int32_t* user; const int32_t* item;
  const double* theta; const double* eta; const double* pr;
  double* rat;          // [S][M][R]
  int64_t M;
  int U, I, R, K, L, ldk, ldl;
};

// SMEM_P: pr staged in shared memory as [R][K][L]; otherwise (tables too large for shared memory)
// read in place from global memory, where it stays L2-resident.  Same products, same order.
template <bool SMEM_P>
__global__ void __launch_bounds__(256) prod_dist_kernel(const ProdArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = A.K, L = A.L, R = A.R;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int run = blockIdx.y;
  const double* prs = A.pr + (size_t)run * K * L * R;
  double* Pq = reinterpret_cast<double*>(smem_raw);          // [R][K][L] (SMEM_P)
  double* th_s = SMEM_P ? Pq + (size_t)R * K * L : Pq;       // [warps][K]
  if (SMEM_P) {
    for (int t = threadIdx.x; t < K * L * R; t += blockDim.x) {
      int kl = t / R, r = t - kl * R;
      Pq[(size_t)r * K * L + kl] = __ldg(prs + t);
    }
  }
  __syncthreads();
  double* th = th_s + warp * K;
  const double* theta_run = A.theta + (size_t)run * A.U * A.ldk;
  const double* eta_run = A.eta + (size_t)run * A.I * A.ldl;
  for (int64_t m = (int64_t)blockIdx.x * nwarp + warp; m < A.M; m += (int64_t)gridDim.x * nwarp) {
    const int u = __ldg(A.user + m), it = __ldg(A.item + m);
    MMSBM_DEV_CHECK(u >= 0 && u < A.U && it >= 0 && it < A.I);
    __syncwarp();
    for (int k = lane; k < K; k += 32) th[k] = __ldg(theta_run + (size_t)u * A.ldk + k);
    __syncwarp();
    const double* erow = eta_run + (size_t)it * A.ldl;
    for (int r = 0; r < R; ++r) {
      const double* Pr = SMEM_P ? Pq + (size_t)r * K * L : prs + r;
      double acc = 0.0;
      for (int l0 = 0; l0 < L; l0 += 32) {
        const int l = l0 + lane;
        if (l < L) {
          const double e = __ldg(erow + l);
          for (int k = 0; k < K; ++k) {
            const double p = SMEM_P ? Pr[k * L + l] : __ldg(Pr + (size_t)(k * L + l) * R);
            acc = fma(th[k] * e, p, acc);
          }
        }
      }
      acc = warp_sum(acc);
      if (lane == 0) A.rat[((size_t)run * A.M + m) * R + r] = acc;
    }
  }
}

// ---- prediction statistics -----------------------------------------------------------------
struct StatArgs {
  const double* rat; const int32_t* real;
  int64_t M; int R;
  int64_t* cnt_partial;   // [S][blocks][5]
  double* s2_partial;     // [S][blocks]
  int32_t* pred;          // [S][M] or null
};

__global__ void __launch_bounds__(256) stats_kernel(const StatArgs A) {
  __shared__ long long c_s[256][5];
  __shared__ double d_s[256];
  const int run = blockIdx.y;
  long long c[5] = {0, 0, 0, 0, 0};
  double s2p = 0.0;
  for (int64_t m = (int64_t)blockIdx.x * 256 + threadIdx.x; m < A.M; m += (int64_t)gridDim.x * 256) {
    const double* row = A.rat + ((size_t)run * A.M + m) * A.R;
    double best = row[0], tot = 0.0, expect = 0.0;
    int arg = 0;
    for (int r = 0; r < A.R; ++r) {
      const double v = row[r];
      if (v > best) { best = v; arg = r; }   // first maximum, as np.argmax
      tot += v;
      expect = fma(v, (double)r, expect);    // rat @ [0..R-1]  (src/mmsbm.py:518)
    }
    if (A.pred) A.pred[(size_t)run * A.M + m] = arg;
    if (tot != 0.0) {                        // rows with an all-zero distribution are dropped
      const int real = A.real[m];
      const int gap = abs(arg - real);
      c[0] += 1;
      c[1] += (gap == 0);
      c[2] += (gap <= 1);
      c[3] += gap;
      c[4] += ((double)real == rint(expect));  // np.round: half to even
      s2p += fabs(expect - (double)real);
    }
  }
  for (int k = 0; k < 5; ++k) c_s[threadIdx.x][k] = c[k];
  d_s[threadIdx.x] = s2p;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      for (int k = 0; k < 5; ++k) c_s[threadIdx.x][k] += c_s[threadIdx.x + s][k];
      d_s[threadIdx.x] += d_s[threadIdx.x + s];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const size_t b = (size_t)run * gridDim.x + blockIdx.x;
    for (int k = 0; k < 5; ++k) A.cnt_partial[b * 5 + k] = c_s[0][k];
    A.s2_partial[b] = d_s[0];
  }
}

__global__ void stats_final_kernel(const int64_t* cnt_partial, const double* s2_partial, int blocks,
                                   int64_t* counts, double* s2pond) {
  const int run = blockIdx.x;
  if (threadIdx.x < 5) {
    long long acc = 0;
    for (int b = 0; b < blocks; ++b) acc += cnt_partial[((size_t)run * blocks + b) * 5 + threadIdx.x];
    counts[run * 5 + threadIdx.x] = acc;
  } else if (threadIdx.x == 5) {
    double acc = 0.0;
    for (int b = 0; b < blocks; ++b) acc += s2_partial[(size_t)run * blocks + b];
    s2pond[run] = acc;
  }
}

__global__ void mean_runs_kernel(const double* rat, int64_t n, int S, double* mean) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  double acc = rat[t];
  for (int s = 1; s < S; ++s) acc += rat[(size_t)s * n + t];   // slab order, as np.mean(axis=0)
  mean[t] = acc / (double)S;
}

__global__ void omegas_kernel(const int32_t* user, const int32_t* item, const int32_t* level,
                              int64_t total, int K, int L, int R, int ldk, int ldl,
                              const double* theta, const double* eta, const double* pr, double* out) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const int KL = K * L;
  const int64_t n = t / KL;
  const int kl = (int)(t - n * KL), k = kl / L, l = kl - k * L;
  const int u = user[n], i = item[n], r = level[n];
  // (theta * eta) * pr, the reference's left-to-right product (src/kernels_numpy.py:32-36)
  out[t] = __dmul_rn(__dmul_rn(theta[(size_t)u * ldk + k], eta[(size_t)i * ldl + l]),
                     pr[(size_t)kl * R + r]);
}

constexpr int kStatBlocks = 296;

}  // namespace mmsbm

using namespace mmsbm;

// [2][R][K][L] tables of one run of the element-wise likelihood (global memory when they do not fit
// shared memory)
static size_t lik_table_bytes(int R, int K, int L) { return 2 * (size_t)R * K * L * 8; }
// the element-wise kernel keeps its two tables in global memory when they and the theta rows of its
// warps do not fit 200 KB of shared memory
static size_t lik_elementwise_smem(int R, int K, int L) { return (2 * (size_t)R * K * L + 2 * (size_t)kLikWarps * K) * 8; }
static bool lik_elementwise_tables(int R, int K, int L) { return lik_elementwise_smem(R, K, L) > 200 * 1024; }
// what the element-wise evaluation takes from the workspace (partials, and tables when it needs them)
static size_t lik_elementwise_bytes(int R, int K, int L, int S) {
  return align_up((size_t)S * kLikCtas * kLikWarps * 8) +
         (lik_elementwise_tables(R, K, L) ? align_up((size_t)S * lik_table_bytes(R, K, L)) : 0);
}

static int lik_env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

// the factorised path needs rows of at most 32 doubles (one 32-byte chunk per lane of a group of
// up to 8) and both operand tables of a run in shared memory
static bool lik_factorised_ok(int R, int K, int L) {
  const int ldk = row_stride(K), ldl = row_stride(L);
  return ldk <= 32 && ldl <= 32 && 2 * (size_t)ldk * R * ldl * 8 <= 200 * 1024 &&
         lik_env_int("MMSBM_LIK_ELEMENTWISE", 0) == 0;
}
static size_t lik_run_bytes(int U, int I, int R, int L) {      // tables of one run
  const size_t ldl = row_stride(L), rnb = (size_t)R * ldl;
  return 2 * align_up((size_t)U * rnb * 8) + align_up((size_t)I * 2 * ldl * 8);
}
static int64_t lik_pmax(int64_t N, int U) { return (int64_t)U + N / MMSBM_PIECE_LEN + 1; }   // = graph_build.cu
// the factorised path's fixed part: two partials per piece, the per-run |log S~| sum and redo flag,
// and room for the element-wise evaluation of the runs it hands over.  Its tables are usually in
// shared memory, but not always: K = 16, L = 32, R = 25 passes lik_factorised_ok (16 R ldk ldl =
// 200 KB) while the element-wise kernel also needs 2 K doubles per warp.
static size_t lik_fact_fixed_bytes(int64_t N, int U, int R, int K, int L, int S) {
  return 2 * align_up((size_t)S * lik_pmax(N, U) * 8) + align_up((size_t)S * 8) + align_up((size_t)S * 4) +
         lik_elementwise_bytes(R, K, L, S);
}

extern "C" int mmsbm_likelihood_workspace_bytes(int64_t N, int32_t U, int32_t I, int32_t R, int32_t K,
                                                int32_t L, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_likelihood_workspace_bytes: bad argument");
  const size_t elementwise = lik_elementwise_bytes(R, K, L, S) + 256;
  size_t fact = 0;
  if (lik_factorised_ok(R, K, L))
    fact = lik_fact_fixed_bytes(N, U, R, K, L, S) + (size_t)S * lik_run_bytes(U, I, R, L) + 256;
  *bytes = fact > elementwise ? fact : elementwise;
  return 0;
}

// smallest workspace mmsbm_likelihood accepts: the runs are then processed one at a time
extern "C" int mmsbm_likelihood_min_workspace_bytes(int64_t N, int32_t U, int32_t I, int32_t R, int32_t K,
                                                    int32_t L, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_likelihood_min_workspace_bytes: bad argument");
  const size_t elementwise = lik_elementwise_bytes(R, K, L, S) + 256;
  size_t fact = 0;
  if (lik_factorised_ok(R, K, L))
    fact = lik_fact_fixed_bytes(N, U, R, K, L, S) + lik_run_bytes(U, I, R, L) + 256;
  *bytes = fact > elementwise ? fact : elementwise;
  return 0;
}

// Element-wise form: K*L visits per rating, partials and (when they do not fit shared memory)
// tables taken from the arena.  With redo, only the runs flagged there are evaluated and written.
static int likelihood_elementwise(Arena& arena, const int32_t* useg, const int32_t* uadj, int U, int I, int R,
                                  int K, int L, int S, const double* theta, const double* eta, const double* pr,
                                  double* out, const int* redo, cudaStream_t st) {
  const int nw = kLikCtas * kLikWarps;
  double* partial = arena.take<double>((size_t)S * nw);
  MMSBM_REQUIRE(partial, MMSBM_ENOMEM, "mmsbm_likelihood: workspace too small");
  LikArgs a{useg, uadj, theta, eta, pr, partial, nullptr, U, I, R, K, L, row_stride(K), row_stride(L), redo};
  size_t smem = lik_elementwise_smem(R, K, L);
  if (lik_elementwise_tables(R, K, L)) {         // keep the two tables in global memory (L2 resident)
    a.tables = arena.take<double>((size_t)S * lik_table_bytes(R, K, L) / 8);
    MMSBM_REQUIRE(a.tables, MMSBM_ENOMEM, "mmsbm_likelihood: workspace too small");
    const int n = K * L * R;
    lik_tables_kernel<<<dim3((n + 255) / 256, S), 256, 0, st>>>(pr, K, L, R, a.tables, redo);
    MMSBM_LAUNCH_CHECK("lik_tables_kernel");
    smem = 2 * (size_t)kLikWarps * K * 8;
  }
  MMSBM_CUDA(cudaFuncSetAttribute(likelihood_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  likelihood_kernel<<<dim3(kLikCtas, S), kLikWarps * 32, smem, st>>>(a);
  MMSBM_LAUNCH_CHECK("likelihood_kernel");
  sum_partials_kernel<<<S, 256, 0, st>>>(partial, nw, out, redo);
  MMSBM_LAUNCH_CHECK("sum_partials_kernel");
  return 0;
}

template <int LD>
static int launch_lik_tables(const double* theta, const double* pr, double* W, double* A, int U, int K, int L,
                             int R, int run0, int nb, cudaStream_t st) {
  const int ldl = row_stride(L);
  const size_t smem = 2 * (size_t)LD * R * ldl * 8;
  MMSBM_CUDA(cudaFuncSetAttribute(lik_user_tables_kernel<LD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int gx = (U + 255) / 256 < sm_count() * 2 ? (U + 255) / 256 : sm_count() * 2;
  lik_user_tables_kernel<LD><<<dim3(gx, nb), 256, smem, st>>>(theta, pr, W, A, U, K, L, R, ldl, run0);
  MMSBM_LAUNCH_CHECK("lik_user_tables_kernel");
  return 0;
}

static int likelihood_factorised(const int32_t* useg, const int32_t* uadj, const int32_t* usched, int64_t N,
                                 int U, int I, int R, int K, int L, int S, const double* theta,
                                 const double* eta, const double* pr, double* out, void* ws, size_t ws_bytes,
                                 cudaStream_t st) {
  const int ldk = row_stride(K), ldl = row_stride(L);
  const size_t rnb = (size_t)R * ldl;
  const int64_t pmax = lik_pmax(N, U);
  MMSBM_REQUIRE(pmax <= 0x7fffffff, MMSBM_ERANGE, "mmsbm_likelihood: too many pieces");
  Arena arena(ws, ws_bytes);
  double* partial = arena.take<double>((size_t)S * pmax);
  double* lpartial = arena.take<double>((size_t)S * pmax);
  double* labs = arena.take<double>(S);
  int* redo = arena.take<int>(S);
  MMSBM_REQUIRE(partial && lpartial && labs && redo, MMSBM_ENOMEM, "mmsbm_likelihood: workspace too small");
  const size_t per_run = lik_run_bytes(U, I, R, L), reserved = lik_elementwise_bytes(R, K, L, S);
  // runs per batch that fit the workspace next to what the element-wise evaluation takes
  int nb = ws_bytes - arena.off >= reserved ? (int)((ws_bytes - arena.off - reserved) / per_run) : 0;
  if (nb > S) nb = S;
  MMSBM_REQUIRE(nb >= 1, MMSBM_ENOMEM, "mmsbm_likelihood: workspace too small for one run (%zu bytes)", ws_bytes);
  double* W = arena.take<double>((size_t)nb * U * rnb);
  double* A = arena.take<double>((size_t)nb * U * rnb);
  double* e2 = arena.take<double>((size_t)nb * I * 2 * ldl);
  MMSBM_REQUIRE(W && A && e2, MMSBM_ENOMEM, "mmsbm_likelihood: workspace too small");
  MMSBM_CUDA(cudaMemsetAsync(partial, 0, (size_t)S * pmax * 8, st));
  MMSBM_CUDA(cudaMemsetAsync(lpartial, 0, (size_t)S * pmax * 8, st));
  for (int run0 = 0; run0 < S; run0 += nb) {
    const int n = S - run0 < nb ? S - run0 : nb;
    {
      const size_t rows = (size_t)n * I, tot = rows * ldl;
      lik_eta_table_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(eta + (size_t)run0 * I * ldl, e2, rows, ldl);
      MMSBM_LAUNCH_CHECK("lik_eta_table_kernel");
    }
    int rc = MMSBM_ERANGE;
    switch (ldk) {
      case 4: rc = launch_lik_tables<4>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 8: rc = launch_lik_tables<8>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 12: rc = launch_lik_tables<12>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 16: rc = launch_lik_tables<16>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 20: rc = launch_lik_tables<20>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 24: rc = launch_lik_tables<24>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 28: rc = launch_lik_tables<28>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
      case 32: rc = launch_lik_tables<32>(theta, pr, W, A, U, K, L, R, run0, n, st); break;
    }
    if (rc) return rc;
    LikPassArgs a{useg, uadj, usched, e2, W, A, partial + (size_t)run0 * pmax, pmax, U, I, R, ldl,
                  lpartial + (size_t)run0 * pmax};
    const int64_t want = (pmax + 7) / 8;
    const int64_t cap = (int64_t)sm_count() * 16;
    const dim3 grid((unsigned)(want < cap ? want : cap), n);
    switch (ldl / 4) {
      case 1: lik_pass_kernel<1><<<grid, 256, 0, st>>>(a); break;
      case 2: lik_pass_kernel<2><<<grid, 256, 0, st>>>(a); break;
      case 3: lik_pass_kernel<3><<<grid, 256, 0, st>>>(a); break;
      case 4: lik_pass_kernel<4><<<grid, 256, 0, st>>>(a); break;
      case 5: lik_pass_kernel<5><<<grid, 256, 0, st>>>(a); break;
      case 6: lik_pass_kernel<6><<<grid, 256, 0, st>>>(a); break;
      case 7: lik_pass_kernel<7><<<grid, 256, 0, st>>>(a); break;
      default: lik_pass_kernel<8><<<grid, 256, 0, st>>>(a); break;
    }
    MMSBM_LAUNCH_CHECK("lik_pass_kernel");
  }
  sum_partials_kernel<<<S, 256, 0, st>>>(partial, (int)pmax, out);
  MMSBM_LAUNCH_CHECK("sum_partials_kernel");
  sum_partials_kernel<<<S, 256, 0, st>>>(lpartial, (int)pmax, labs);
  MMSBM_LAUNCH_CHECK("sum_partials_kernel");
  lik_check_kernel<<<(S + 127) / 128, 128, 0, st>>>(out, labs, S, (double)K * L * kEps, -2.0 * (double)N * log(kEps),
                                                     redo);
  MMSBM_LAUNCH_CHECK("lik_check_kernel");
  // the runs the bound does not clear: the element-wise form, whose bits replace the factorised total
  return likelihood_elementwise(arena, useg, uadj, U, I, R, K, L, S, theta, eta, pr, out, redo, st);
}

extern "C" int mmsbm_likelihood(const int32_t* useg, const int32_t* uadj, const int32_t* usched, int64_t N,
                                int32_t U, int32_t I, int32_t R, int32_t K, int32_t L, int32_t S,
                                const double* theta, const double* eta, const double* pr, double* out,
                                void* ws, size_t ws_bytes, void* stream) {
  MMSBM_REQUIRE(useg && uadj && theta && eta && pr && out && ws, MMSBM_EINVAL,
                "mmsbm_likelihood: null pointer");
  MMSBM_REQUIRE(U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0 && N >= 0, MMSBM_EINVAL,
                "mmsbm_likelihood: bad size");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (usched && lik_factorised_ok(R, K, L))
    return likelihood_factorised(useg, uadj, usched, N, U, I, R, K, L, S, theta, eta, pr, out, ws, ws_bytes, st);
  // element-wise path (rows wider than 32 doubles, or no schedule given)
  Arena arena(ws, ws_bytes);
  return likelihood_elementwise(arena, useg, uadj, U, I, R, K, L, S, theta, eta, pr, out, nullptr, st);
}

// ---- observed-data log-likelihood ----------------------------------------------------------
// l = sum_n log max(S_n, eps), S_n = sum_kl theta_uk eta_il p_klr = <W_{u,r}, eta_i>: the EM
// objective (it never decreases from one EM step to the next).  W = theta x Pw comes from the EM
// step's own contraction (prep_p_kernel + launch_w, every admitted shape); the by-user pass of the
// factorised likelihood then gathers one eta row per rating, with the same piece schedule and the
// same fixed-order two-stage sum.  All runs at once.
static size_t loglik_bytes(int64_t N, int U, int R, int K, int L, int S) {
  const size_t ldk = row_stride(K), ldl = row_stride(L);
  return 4 * align_up((size_t)S * ldk * ldl * R * 8) + align_up((size_t)S * U * R * ldl * 8) +
         align_up((size_t)S * lik_pmax(N, U) * 8) + 256;
}

namespace mmsbm {
int launch_loglik(const int32_t* useg, const int32_t* uadj, const int32_t* usched, int64_t N, int U, int I,
                  int R, int K, int L, int S, const double* theta, const double* eta, const double* pr,
                  double* out, void* ws, size_t ws_bytes, cudaStream_t st) {
  const int ldk = row_stride(K), ldl = row_stride(L), rnb = R * ldl;
  const int64_t pmax = lik_pmax(N, U);
  MMSBM_REQUIRE(pmax <= 0x7fffffff, MMSBM_ERANGE, "mmsbm_loglik: too many pieces");
  Arena arena(ws, ws_bytes);
  const size_t p_elems = (size_t)S * ldk * ldl * R;
  double* pw = arena.take<double>(p_elems);                  // user-side operand layout (the one used)
  double* pn = arena.take<double>(p_elems);
  double* pwi = arena.take<double>(p_elems);
  double* pni = arena.take<double>(p_elems);
  double* W = arena.take<double>((size_t)S * U * rnb);
  double* partial = arena.take<double>((size_t)S * pmax);
  MMSBM_REQUIRE(pw && pn && pwi && pni && W && partial, MMSBM_ENOMEM, "mmsbm_loglik: workspace too small (%zu)",
                ws_bytes);
  int rc;
  if ((rc = launch_prep_p(pr, K, L, R, ldk, ldl, S, pw, pn, pwi, pni, st))) return rc;
  if ((rc = launch_w(theta, pw, W, U, ldk, rnb, S, st))) return rc;
  MMSBM_CUDA(cudaMemsetAsync(partial, 0, (size_t)S * pmax * 8, st));
  LikPassArgs a{useg, uadj, usched, eta, W, nullptr, partial, pmax, U, I, R, ldl};
  const int64_t want = (pmax + 7) / 8;
  const int64_t cap = (int64_t)sm_count() * 16;
  const dim3 grid((unsigned)(want < cap ? want : cap), S);
  switch (ldl < 32 ? ldl / 4 : 8) {
    case 1: loglik_pass_kernel<1><<<grid, 256, 0, st>>>(a); break;
    case 2: loglik_pass_kernel<2><<<grid, 256, 0, st>>>(a); break;
    case 3: loglik_pass_kernel<3><<<grid, 256, 0, st>>>(a); break;
    case 4: loglik_pass_kernel<4><<<grid, 256, 0, st>>>(a); break;
    case 5: loglik_pass_kernel<5><<<grid, 256, 0, st>>>(a); break;
    case 6: loglik_pass_kernel<6><<<grid, 256, 0, st>>>(a); break;
    case 7: loglik_pass_kernel<7><<<grid, 256, 0, st>>>(a); break;
    default: loglik_pass_kernel<8><<<grid, 256, 0, st>>>(a); break;
  }
  MMSBM_LAUNCH_CHECK("loglik_pass_kernel");
  sum_partials_kernel<<<S, 256, 0, st>>>(partial, (int)pmax, out);
  MMSBM_LAUNCH_CHECK("sum_partials_kernel");
  return 0;
}
}  // namespace mmsbm

extern "C" int mmsbm_loglik_workspace_bytes(int64_t N, int32_t U, int32_t I, int32_t R, int32_t K, int32_t L,
                                            int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && N >= 0 && U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0, MMSBM_EINVAL,
                "mmsbm_loglik_workspace_bytes: bad argument");
  *bytes = loglik_bytes(N, U, R, K, L, S);
  return 0;
}

extern "C" int mmsbm_loglik(const int32_t* useg, const int32_t* uadj, const int32_t* usched, int64_t N,
                            int32_t U, int32_t I, int32_t R, int32_t K, int32_t L, int32_t S,
                            const double* theta, const double* eta, const double* pr, double* out,
                            void* ws, size_t ws_bytes, void* stream) {
  MMSBM_REQUIRE(useg && uadj && usched && theta && eta && pr && out && ws, MMSBM_EINVAL,
                "mmsbm_loglik: null pointer");
  MMSBM_REQUIRE(U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0 && N >= 0, MMSBM_EINVAL,
                "mmsbm_loglik: bad size");
  MMSBM_REQUIRE(K <= 256 && L <= 256 && R <= 31, MMSBM_ERANGE,
                "mmsbm_loglik: K, L <= 256 and R <= 31 supported (K=%d L=%d R=%d)", K, L, R);
  return launch_loglik(useg, uadj, usched, N, U, I, R, K, L, S, theta, eta, pr, out, ws, ws_bytes,
                       static_cast<cudaStream_t>(stream));
}

extern "C" int mmsbm_prod_dist(const int32_t* user, const int32_t* item, int64_t M, int32_t U,
                               int32_t I, int32_t R, int32_t K, int32_t L, int32_t S,
                               const double* theta, const double* eta, const double* pr, double* rat,
                               void* stream) {
  MMSBM_REQUIRE(theta && eta && pr && (M == 0 || (user && item && rat)), MMSBM_EINVAL,
                "mmsbm_prod_dist: null pointer");
  MMSBM_REQUIRE(U > 0 && I > 0 && R > 0 && K > 0 && L > 0 && S > 0 && M >= 0, MMSBM_EINVAL,
                "mmsbm_prod_dist: bad size");
  if (M == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProdArgs a{user, item, theta, eta, pr, rat, M, U, I, R, K, L, row_stride(K), row_stride(L)};
  const size_t th_bytes = 8 * (size_t)K * 8;                 // theta rows of the 8 warps
  size_t smem = (size_t)R * K * L * 8 + th_bytes;
  const bool smem_p = smem <= kMaxSmemBytes;
  if (!smem_p) smem = th_bytes;
  auto kern = smem_p ? prod_dist_kernel<true> : prod_dist_kernel<false>;
  MMSBM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t want = (M + 7) / 8;
  const int64_t cap = (int64_t)sm_count() * 8;
  unsigned grid = (unsigned)(want < cap ? want : cap);
  kern<<<dim3(grid, S), 256, smem, st>>>(a);
  MMSBM_LAUNCH_CHECK("prod_dist_kernel");
  return 0;
}

extern "C" int mmsbm_stats_workspace_bytes(int64_t M, int32_t S, size_t* bytes) {
  MMSBM_REQUIRE(bytes && M >= 0 && S > 0, MMSBM_EINVAL, "mmsbm_stats_workspace_bytes: bad argument");
  *bytes = align_up((size_t)S * kStatBlocks * 5 * 8) + align_up((size_t)S * kStatBlocks * 8) + 256;
  return 0;
}

extern "C" int mmsbm_predict_stats(const double* rat, const int32_t* real, int64_t M, int32_t R,
                                   int32_t S, int64_t* counts, double* s2pond, int32_t* pred, void* ws,
                                   size_t ws_bytes, void* stream) {
  MMSBM_REQUIRE(counts && s2pond && ws && (M == 0 || (rat && real)), MMSBM_EINVAL,
                "mmsbm_predict_stats: null pointer");
  MMSBM_REQUIRE(M >= 0 && R > 0 && S > 0, MMSBM_EINVAL, "mmsbm_predict_stats: bad size");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Arena arena(ws, ws_bytes);
  int64_t* cp = arena.take<int64_t>((size_t)S * kStatBlocks * 5);
  double* sp = arena.take<double>((size_t)S * kStatBlocks);
  MMSBM_REQUIRE(cp && sp, MMSBM_ENOMEM, "mmsbm_predict_stats: workspace too small");
  StatArgs a{rat, real, M, R, cp, sp, pred};
  stats_kernel<<<dim3(kStatBlocks, S), 256, 0, st>>>(a);
  MMSBM_LAUNCH_CHECK("stats_kernel");
  stats_final_kernel<<<S, 32, 0, st>>>(cp, sp, kStatBlocks, counts, s2pond);
  MMSBM_LAUNCH_CHECK("stats_final_kernel");
  return 0;
}

extern "C" int mmsbm_mean_over_runs(const double* rat, int64_t n, int32_t S, double* mean, void* stream) {
  MMSBM_REQUIRE((n == 0 || (rat && mean)) && n >= 0 && S > 0, MMSBM_EINVAL, "mmsbm_mean_over_runs: bad argument");
  if (n == 0) return 0;
  mean_runs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(rat, n, S, mean);
  MMSBM_LAUNCH_CHECK("mean_runs_kernel");
  return 0;
}

extern "C" int mmsbm_compute_omegas(const int32_t* user, const int32_t* item, const int32_t* level,
                                    int64_t N, int32_t K, int32_t L, int32_t R, const double* theta,
                                    const double* eta, const double* pr, double* omegas, void* stream) {
  MMSBM_REQUIRE(theta && eta && pr && (N == 0 || (user && item && level && omegas)), MMSBM_EINVAL,
                "mmsbm_compute_omegas: null pointer");
  MMSBM_REQUIRE(N >= 0 && K > 0 && L > 0 && R > 0, MMSBM_EINVAL, "mmsbm_compute_omegas: bad size");
  if (N == 0) return 0;
  const int64_t total = N * K * L;
  omegas_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      user, item, level, total, K, L, R, row_stride(K), row_stride(L), theta, eta, pr, omegas);
  MMSBM_LAUNCH_CHECK("omegas_kernel");
  return 0;
}
