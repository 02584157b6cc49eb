// Whole EM fits of SMALL problems (one run, rows of at most 12 doubles, up to a few million
// ratings: BASELINE.json's ML-100K configuration) in ONE cooperative kernel launch.
//
// At this size an iteration of em_step.cu is a chain of dependent kernels of a few microseconds
// each (0.051 ms for 11 launches even as a replayed CUDA graph): launch latency, not work, sets
// the pace.  Here the loop over the iterations runs INSIDE the kernel and the stages of an
// iteration are separated by two grid-wide barriers instead of launches:
//
//   every warp   segments (users and items alike, dealt statically: segment s belongs to CTA
//                s mod gridDim.x, warp (s / gridDim.x) mod 8): w = own x P from shared memory
//                (no W table), the ratings level by level (G lanes per neighbour row, one
//                256-bit load per lane, the same factorised algebra as segment_pass.cuh), then
//                own' = own o (g x P) / max(deg, 1) straight into the next parameter buffer (no G
//                table) and, on the emitting side, the rank-1 update own (x) g into per-lane
//                register accumulators of n_pr.  A segment with more than kSmallLong ratings is
//                walked by all eight warps of its CTA together
//   CTA          accumulators added in warp order -> one partial n_pr per CTA       | grid barrier
//   warp / (k,l) partial sums over the CTAs in a fixed order, x P, normalise over r | grid barrier
//
// Both parameter sets are double buffered (an iteration reads buffer `it & 1`, writes the other),
// so users and items are processed in the same phase.  Every sum has a fixed order for a fixed
// grid: results are reproducible; against em_step.cu they differ in the last bits (different
// association), which is why the path is chosen by the SHAPE alone, never by the iteration count.
// Replaces the loop src/mmsbm.py:243-250 for such shapes; MMSBM_COOP=0 turns it off.
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"
#include "em_internal.cuh"
#include "segment_pass.cuh"

namespace cg = cooperative_groups;

namespace mmsbm {

constexpr int kSmallWarps = 12;     // per CTA, one CTA per SM: 170 registers per thread
constexpr int kSmallLong = 1024;      // longer segments are walked by a whole CTA
constexpr int kSmallMaxR = 8;

struct SmallArgs {
  const int32_t* seg[2];              // [0] users: useg, [1] items: iseg      [n*R + 1]
  const int32_t* adj[2];              // neighbour ids (users: items, items: users)
  const int32_t* deg[2];
  double* own[2][2];                  // own[side][buffer]: theta / eta, [n][LD]
  double* pr[2];                      // [K][L][R]
  double* partial;                    // [gridDim.x][R*LD*LD]
  int n[2];                           // U, I
  int R, K, L, iterations, emit_side;
};

// theta / eta / pr are WRITTEN by this kernel (another CTA, the previous iteration): they must be read with
// ordinary coherent loads -- the read-only path (ld.global.nc, __ldg) is outside the memory model and
// may serve a stale line after the grid barrier.  The index arrays are read-only for the whole launch.
__device__ __forceinline__ double4_t ld256_coherent(const double* p) {
  double4_t v;
  asm volatile("ld.global.v4.f64 {%0,%1,%2,%3}, [%4];"
               : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p) : "memory");
  return v;
}

// P[r][k][l] in shared memory as the side sees it: a = own index, b = neighbour index
__device__ __forceinline__ double p_at(const double* Ps, int LD, int side, int r, int a, int b) {
  return side == 0 ? Ps[(r * LD + a) * LD + b] : Ps[(r * LD + b) * LD + a];
}

template <int LD>
__global__ void __launch_bounds__(kSmallWarps * 32, 1) em_small_kernel(const SmallArgs A) {
  cg::grid_group grid = cg::this_grid();
  constexpr int G = LD / 4;                     // lanes per neighbour row
  constexpr int RPS = 32 / G;                   // ratings per step
  constexpr int UN = (G == 1) ? 1 : (G == 2) ? 2 : 3;   // steps per chunk (UN * RPS <= 32 ids per chunk)
  constexpr int SLOTS = UN * RPS;
  const int R = A.R, NE = R * LD * LD, RLD = R * LD;

  extern __shared__ __align__(32) unsigned char smem_raw[];
  double* Ps = reinterpret_cast<double*>(smem_raw);          // [R][LD][LD]
  double* warp_area = Ps + NE;              // per warp: own_s[LD] | w_s[R*LD] | g_s[R*LD] | acc_s[NE] (n_pr accumulators)
  __shared__ int long_side[kSmallWarps], long_id[kSmallWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int per_warp = LD + 2 * RLD + NE;
  double* own_s = warp_area + (size_t)warp * per_warp;
  double* w_s = own_s + LD;
  double* g_s = w_s + RLD;
  double* acc_s = g_s + RLD;
  const int grp = lane / G, q = lane - grp * G;
  const bool lane_on = grp < RPS;
  const GroupSum<G> group_sum(grp * G, q);
  const int nseg = A.n[0] + A.n[1];

  // own row and w = own x P of segment (side, id) into this warp's shared memory
  auto load_own_and_w = [&](int side, int id, int cur) {
    const double* row = A.own[side][cur] + (size_t)id * LD;
    if (lane < LD) own_s[lane] = row[lane];
    __syncwarp();
    for (int v = lane; v < RLD; v += 32) {
      const int r = v / LD, b = v - r * LD;
      double s = 0.0;
#pragma unroll
      for (int a = 0; a < LD; ++a) s = fma(own_s[a], p_at(Ps, LD, side, r, a, b), s);
      w_s[v] = s;
    }
    __syncwarp();
  };

  // g_r of the ratings [lo_r, hi_r) of every level r (part `part` of `nparts` of each level's range)
  // -> this warp's g_s
  auto stream_levels = [&](int side, int id, int cur, int part, int nparts) {
    const int32_t* seg = A.seg[side] + (size_t)id * R;
    const int32_t* adj = A.adj[side];
    const double* nbr = A.own[side ^ 1][cur];
    // the first chunk of ids of every level, loaded back to back (one latency for all levels)
    int lo_r[kSmallMaxR], hi_r[kSmallMaxR], first_ids[kSmallMaxR];
#pragma unroll
    for (int r = 0; r < kSmallMaxR; ++r) {
      lo_r[r] = hi_r[r] = 0; first_ids[r] = 0;
      if (r < R) {
        const int b = __ldg(seg + r), e = __ldg(seg + r + 1), len = e - b;
        lo_r[r] = b + (int)(((int64_t)len * part) / nparts);
        hi_r[r] = b + (int)(((int64_t)len * (part + 1)) / nparts);
      }
    }
#pragma unroll
    for (int r = 0; r < kSmallMaxR; ++r)
      if (r < R && lane < SLOTS && lo_r[r] + lane < hi_r[r]) first_ids[r] = ld_stream(adj + lo_r[r] + lane);
#pragma unroll
    for (int r = 0; r < kSmallMaxR; ++r) {
      if (r >= R) break;
      double4_t g{0.0, 0.0, 0.0, 0.0};
      const double4_t wr = lane_on ? lds32(w_s + r * LD + 4 * q) : double4_t{0.0, 0.0, 0.0, 0.0};
      int ids = first_ids[r];
      for (int pos = lo_r[r]; pos < hi_r[r]; pos += SLOTS) {
        const int cnt = min(SLOTS, hi_r[r] - pos);
        double4_t x[UN];
        bool valid[UN];
#pragma unroll
        for (int un = 0; un < UN; ++un) {
          const int sl = un * RPS + grp;
          int nid = __shfl_sync(kFull, ids, sl & 31);
          valid[un] = lane_on && sl < cnt;
          if (!valid[un]) nid = 0;                           // row 0: in bounds, weight zero
          MMSBM_DEV_CHECK(nid >= 0 && nid < A.n[side ^ 1]);
          x[un] = ld256_coherent(nbr + (size_t)nid * LD + 4 * q);
        }
        {                                                    // ids of the next chunk of this level
          const int nxt = pos + SLOTS + lane;
          ids = (lane < SLOTS && nxt < hi_r[r]) ? ld_stream(adj + nxt) : 0;
        }
#pragma unroll
        for (int un = 0; un < UN; ++un) {
          double part_sum = fma(x[un].x, wr.x, x[un].y * wr.y);
          part_sum = fma(x[un].z, wr.z, part_sum);
          part_sum = fma(x[un].w, wr.w, part_sum);
          const double tot = group_sum(part_sum);
          const double inv = valid[un] ? rcp_clamped(tot) : 0.0;
          g.x = fma(x[un].x, inv, g.x); g.y = fma(x[un].y, inv, g.y);
          g.z = fma(x[un].z, inv, g.z); g.w = fma(x[un].w, inv, g.w);
        }
      }
      // sum over the RPS groups (fixed order), group 0 stores
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        if (off < RPS) {
          const double tx = __shfl_down_sync(kFull, g.x, off * G), ty = __shfl_down_sync(kFull, g.y, off * G);
          const double tz = __shfl_down_sync(kFull, g.z, off * G), tw = __shfl_down_sync(kFull, g.w, off * G);
          if (grp + off < RPS) { g.x += tx; g.y += ty; g.z += tz; g.w += tw; }
        }
      }
      if (grp == 0) {
        double* dst = g_s + r * LD + 4 * q;
        dst[0] = g.x; dst[1] = g.y; dst[2] = g.z; dst[3] = g.w;
      }
    }
    __syncwarp();
  };

  // own' = own o (g x P) / max(deg, 1) into the next buffer; rank-1 update of the n_pr accumulators
  auto epilogue = [&](int side, int id, int nxt) {
    if (lane < LD) {
      double s = 0.0;
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int b = 0; b < LD; ++b) s = fma(p_at(Ps, LD, side, r, lane, b), g_s[r * LD + b], s);
      double v = s * own_s[lane];
      v = v / (double)max(__ldg(A.deg[side] + id), 1);
      A.own[side][nxt][(size_t)id * LD + lane] = v;
    }
    if (side == A.emit_side) {
      for (int e = lane; e < NE; e += 32) {
        const int r = e / (LD * LD), k = (e / LD) % LD, l = e % LD;
        acc_s[e] = side == 0 ? fma(own_s[k], g_s[r * LD + l], acc_s[e]) : fma(own_s[l], g_s[r * LD + k], acc_s[e]);
      }
    }
    __syncwarp();
  };

  // does any segment of this CTA need the CTA-wide walk?  (if not, its warps never wait for each other)
  const int stride = gridDim.x * kSmallWarps;
  int mine_long = 0;
  for (int s = blockIdx.x + (int)threadIdx.x * (int)gridDim.x; s < nseg; s += (int)blockDim.x * (int)gridDim.x) {
    const int sd = s >= A.n[0] ? 1 : 0;
    if (__ldg(A.deg[sd] + (sd ? s - A.n[0] : s)) > kSmallLong) mine_long = 1;
  }
  const bool cta_has_long = __syncthreads_or(mine_long) != 0;

  for (int it = 0; it < A.iterations; ++it) {
    const int cur = it & 1, nxt = cur ^ 1;
    for (int e = threadIdx.x; e < NE; e += blockDim.x) {     // P of this iteration, zero padded
      const int r = e / (LD * LD), k = (e / LD) % LD, l = e % LD;
      Ps[e] = (k < A.K && l < A.L) ? A.pr[cur][((size_t)k * A.L + l) * R + r] : 0.0;
    }
    for (int e = lane; e < NE; e += 32) acc_s[e] = 0.0;
    __syncthreads();

    // ---- the segments of this CTA, one per warp and round ----
    if (!cta_has_long) {                                     // the common case: every warp walks its own list
      for (int s = blockIdx.x + warp * (int)gridDim.x; s < nseg; s += stride) {
        const int side = s >= A.n[0] ? 1 : 0, id = side ? s - A.n[0] : s;
        load_own_and_w(side, id, cur);
        stream_levels(side, id, cur, 0, 1);
        epilogue(side, id, nxt);
      }
    } else
    for (int s0 = blockIdx.x; s0 < nseg; s0 += stride) {     // CTA-uniform round loop
      const int s = s0 + warp * gridDim.x;
      const bool have = s < nseg;
      int side = 0, id = 0, dg = 0;
      if (have) {
        side = s >= A.n[0] ? 1 : 0;
        id = side ? s - A.n[0] : s;
        dg = __ldg(A.deg[side] + id);
      }
      const bool is_long = have && dg > kSmallLong;
      if (lane == 0) { long_side[warp] = is_long ? side : -1; long_id[warp] = id; }
      __syncthreads();
      if (have && !is_long) {
        load_own_and_w(side, id, cur);
        stream_levels(side, id, cur, 0, 1);
        epilogue(side, id, nxt);
      }
      __syncthreads();
      for (int w = 0; w < kSmallWarps; ++w) {                // long segments of the round: all warps together
        const int ls = long_side[w];
        if (ls < 0) continue;                                // CTA-uniform
        const int lid = long_id[w];
        load_own_and_w(ls, lid, cur);                        // every warp its own copy of own_s / w_s
        stream_levels(ls, lid, cur, warp, kSmallWarps);
        __syncthreads();
        if (warp == 0) {                                     // partial g rows added in warp order
          for (int v = lane; v < RLD; v += 32) {
            double t = g_s[v];
            for (int ww = 1; ww < kSmallWarps; ++ww) t += warp_area[(size_t)ww * per_warp + LD + RLD + v];   // g_s of warp ww
            g_s[v] = t;
          }
          __syncwarp();
          epilogue(ls, lid, nxt);
        }
        __syncthreads();
      }
      __syncthreads();                                       // the round's flags are free again
    }

    // ---- n_pr: accumulators of the warps added in warp order, one partial per CTA ----
    __syncthreads();
    for (int e = threadIdx.x; e < NE; e += blockDim.x) {
      double t = 0.0;
      for (int w = 0; w < kSmallWarps; ++w) t += warp_area[(size_t)w * per_warp + LD + 2 * RLD + e];
      A.partial[(size_t)blockIdx.x * NE + e] = t;
    }
    grid.sync();

    // ---- pr' = P o (sum over the CTAs), normalised over the rating axis: one warp per (k, l) ----
    for (int kl = blockIdx.x * kSmallWarps + warp; kl < A.K * A.L; kl += stride) {
      const int k = kl / A.L, l = kl - k * A.L;
      double mine = 0.0, tot = 0.0;
      for (int r = 0; r < R; ++r) {
        const int e = (r * LD + k) * LD + l;
        double sm = 0.0;
        for (int c = lane; c < (int)gridDim.x; c += 32) sm += A.partial[(size_t)c * NE + e];
        sm = warp_sum(sm);
        const double v = sm * Ps[e];
        tot += v;
        if (lane == r) mine = v;
      }
      const double dd = (tot == 0.0) ? 1.0 : tot;
      if (lane < R) A.pr[nxt][((size_t)k * A.L + l) * R + lane] = mine / dd;
    }
    grid.sync();
  }
}

template <int LD>
static int launch_small(const SmallArgs& a, int ctas_wanted, cudaStream_t st) {
  auto kern = em_small_kernel<LD>;
  const int NE = a.R * LD * LD;
  const size_t smem = ((size_t)NE + (size_t)kSmallWarps * (LD + 2 * a.R * LD + NE)) * 8;
  MMSBM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  MMSBM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSmallWarps * 32, smem));
  if (per_sm < 1) return MMSBM_ERANGE;
  if (per_sm > 1) per_sm = 1;
  int grid = per_sm * sm_count();
  if (grid > ctas_wanted) grid = ctas_wanted;
  if (grid < 1) grid = 1;
  SmallArgs args = a;
  void* params[] = {&args};
  MMSBM_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kern), dim3(grid), dim3(kSmallWarps * 32), params,
                                         smem, st));
  MMSBM_LAUNCH_CHECK("em_small_kernel");
  return 0;
}

// shapes this path serves (one run, equal row strides of at most 12 doubles, few rating levels)
bool em_small_applicable(int64_t N, int R, int K, int L, int S) {
  return S == 1 && row_stride(K) == row_stride(L) && row_stride(K) <= 12 && R <= kSmallMaxR &&
         N <= ((int64_t)1 << 22);
}
// doubles of the per-CTA partial sums the caller provides (a device-independent bound: 512 CTAs)
size_t em_small_partial_elems(int R, int K) { return (size_t)512 * R * row_stride(K) * row_stride(K); }

// MMSBM_ERANGE: shape not served by this path (the caller takes the multi-kernel path)
int launch_em_small(const int32_t* useg, const int32_t* uadj, const int32_t* udeg, const int32_t* iseg,
                    const int32_t* iadj, const int32_t* ideg, const int32_t* usched, const int32_t* isched, int64_t N,
                    int U, int I, int R, int K, int L, int S, int iterations, double* theta_a, double* eta_a,
                    double* pr_a, double* theta_b, double* eta_b, double* pr_b, double* partial, size_t partial_elems,
                    cudaStream_t st, int long_segments) {
  const int ldk = row_stride(K);
  if (!em_small_applicable(N, R, K, L, S) || iterations <= 0 || !partial) return MMSBM_ERANGE;
  if (env_int("MMSBM_COOP", 1) == 0) return MMSBM_ERANGE;
  int dev = 0, coop = 0;
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess || !coop)
    return MMSBM_ERANGE;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return MMSBM_ERANGE;
  if (long_segments > 0) return MMSBM_ERANGE;
  if (long_segments < 0) {
    // a segment of more than MMSBM_PIECE_LEN ratings (heavy-tailed ids) would be walked by one CTA while the
    // rest of the grid waits at the barrier: such problems stay on the multi-kernel path, whose piece
    // schedule spreads the segment over the GPU.  The schedule headers say whether one exists (16 bytes
    // each; the only host synchronisation of the call)
    int32_t hu[4] = {0, 0, 1, 0}, hi[4] = {0, 0, 1, 0};
    MMSBM_CUDA(cudaMemcpyAsync(hu, usched, sizeof(hu), cudaMemcpyDeviceToHost, st));
    MMSBM_CUDA(cudaMemcpyAsync(hi, isched, sizeof(hi), cudaMemcpyDeviceToHost, st));
    MMSBM_CUDA(cudaStreamSynchronize(st));
    if (hu[2] != 0 || hi[2] != 0) return MMSBM_ERANGE;
  }
  SmallArgs a{};
  a.seg[0] = useg; a.seg[1] = iseg; a.adj[0] = uadj; a.adj[1] = iadj; a.deg[0] = udeg; a.deg[1] = ideg;
  a.own[0][0] = theta_a; a.own[0][1] = theta_b; a.own[1][0] = eta_a; a.own[1][1] = eta_b;
  a.pr[0] = pr_a; a.pr[1] = pr_b;
  a.partial = partial;
  a.n[0] = U; a.n[1] = I;
  a.R = R; a.K = K; a.L = L; a.iterations = iterations;
  a.emit_side = (I <= U) ? 1 : 0;
  const int NE = R * ldk * ldk;
  int ctas = (U + I + kSmallWarps - 1) / kSmallWarps;      // one segment per warp at least
  const int64_t room = (int64_t)(partial_elems / (size_t)NE);
  if (ctas > room) ctas = (int)room;
  if (ctas < 1) return MMSBM_ERANGE;
  switch (ldk) {
    case 4: return launch_small<4>(a, ctas, st);
    case 8: return launch_small<8>(a, ctas, st);
    case 12: return launch_small<12>(a, ctas, st);
  }
  return MMSBM_ERANGE;
}

}  // namespace mmsbm
