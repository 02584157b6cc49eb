// The hot kernel of the EM iteration: a warp takes one piece (up to MMSBM_PIECE_LEN ratings) of a
// segment -- a user in the by-user pass, an item in the by-item pass -- and streams its ratings
// level by level.  See em_step.cu for the algebra.
//
// Lane mapping (all compile time): G lanes hold one neighbour row, lane q its 32-byte chunks
// c*G+q (CH of them), each fetched with ONE 256-bit read-only load (LDG.E.ENL2.256).  A warp
// serves RUNS runs at once over rows interleaved in memory ([group][id][RUNS][NBp]), so a rating
// occupies GR = G*RUNS lanes and its gather is one contiguous RUNS*8*NBp-byte read; RPS = 32/GR
// ratings per step, UN steps per chunk of work (SLOTS = UN*RPS ratings).
//
//   S_n   = <w_level, row>      4*CH DFMA per lane + a sum over the G lanes (5 lanes, 3 steps:
//                               one reduce-scatter for the three dots of a chunk, GroupSum::sum3)
//   1/S_n                       MUFU.RCP64H + one third-order correction
//   g    += row / S_n           4*CH DFMA per lane, registers
//   g_level -> global           once per (piece, level): sum over the RPS groups by shuffles
//
// A chunk is computed in phases -- all UN loads, all dots, all reciprocals, all accumulations --
// so that the loads issue back to back; the last chunk of a level is specialised on the number
// of steps that hold ratings.  w comes from the W table (row_w_kernel) through cp.async into
// shared memory (double buffered, the next piece's rows land while this piece runs; single
// buffered for six runs); g overwrites W in place.  Ratings are stored grouped by level and
// chunks never straddle a level boundary, so the level -- hence w -- is warp-uniform in a chunk.
// Pieces are claimed with an atomic counter: launch-wide (persistent CTAs) or per CTA.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace mmsbm {

constexpr int kWarps = 8;       // warps per CTA of the segment pass

struct alignas(16) double4_t { double x, y, z, w; };

// 256-bit read-only load (LDG.E.ENL2.256 on sm_100a): a lane's 32-byte chunk of a row
__device__ __forceinline__ double4_t ldg256(const double* p) {
  double4_t v;
  // (L1::no_allocate measured 4-9 % slower: the few L1 hits -- row 0 of idle slots, hot ids -- pay)
  asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
      : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void stg256(double* p, const double4_t& v) {
  asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w)
               : "memory");
}
__device__ __forceinline__ double4_t lds32(const double* p) {   // two 128-bit shared loads
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  return double4_t{a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// 1/max(x, eps) for x >= 0: MUFU.RCP64H seed r (relative error e ~ 2^-20) refined by one
// third-order step r(1 + e + e^2), error e^3 ~ 2^-60 -> correctly rounded up to ~1 ulp
__device__ __forceinline__ double rcp_clamped(double x) {
  x = (x < kEps) ? kEps : x;
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double e = fma(-x, r, 1.0);
  const double t = fma(e, e, e);
  return fma(r, t, r);
}

struct SegArgs {
  const int32_t* seg;   // [nseg*R+1]
  const int32_t* adj;   // [N] neighbour ids, grouped by (segment, level)
  const int32_t* sched; // work schedule: pieces of <= MMSBM_PIECE_LEN ratings (graph_build.cu)
  const double* nbr;    // RUNS == 1: [S][nnbr][NBp]   RUNS > 1: [groups][nnbr][RUNS][NBp] (runs interleaved)
  double* wg;           // [S][nseg][R*NBp]  in: w   out: g (in place; single-piece segments)
  double* partial;      // [S][smax][R*NBp]  out: g of the pieces of long segments, by slot
  int64_t pmax, lmax, smax;   // capacities: pieces, long segments, slots (graph_build.cu)
  int nseg, nnbr, NBp, R, segs_per_cta;
  int run_base;         // first run of this launch (grid.y counts runs, or groups of RUNS runs)
  int grp_base;         // RUNS > 1: first run group of this launch inside nbr
  int* counters;        // [gridDim.y] zeroed by the host: pieces are claimed across the whole launch
                        // (persistent CTAs); NULL: every CTA owns segs_per_cta consecutive pieces
};

// w rows in shared memory: double buffered (next piece's rows land while this piece runs) for
// one run or a pair per warp, single buffered for wider run groups (6 runs: 77 KB per CTA otherwise)
__host__ __device__ constexpr int w_buffers(int runs) { return runs > 2 ? 1 : 2; }
inline size_t seg_smem_bytes(int R, int NBp, int runs) {
  return (size_t)kWarps * w_buffers(runs) * runs * R * NBp * 8 + 32;
}
constexpr size_t kMaxSmemBytes = 227 * 1024;   // dynamic shared memory of one CTA on sm_100a

// Sum of `part` over the G consecutive lanes of a group, delivered to every lane of the group.
// Power-of-two groups are aligned, so xor shuffles do; otherwise windows of 1, 2, 4 lanes are
// accumulated by rotating inside the group (source lanes (q+1)%G, (q+2)%G, ... of the group).
// Lanes of one group may round differently in the last bit; each stays deterministic.
template <int G>
struct GroupSum {
  int s1, s2, s4, s6;
  int lead, r1, r2, r3;          // G == 5: sources of the three reduce-scatter stages of sum3()
  bool is0, is1, is2, is3, is14, is03;
  __device__ __forceinline__ GroupSum(int leader, int q) {
    s1 = (leader + (q + 1) % G) & 31;
    s2 = (leader + (q + 2) % G) & 31;
    s4 = (leader + (q + 4) % G) & 31;
    s6 = (leader + (q + 6) % G) & 31;
    lead = leader & 31;
    is0 = q == 0; is1 = q == 1; is2 = q == 2; is3 = q == 3; is14 = (q == 1) | (q == 4); is03 = (q == 0) | (q == 3);
    // stage 1: 0<-1 1<-2 2<-0 3<-4 4<-3   stage 2: 0<-2 1<-4 2<-3 4<-0   stage 3: 0<-3 1<-4 2<-1
    r1 = (leader + (q == 0 ? 1 : q == 1 ? 2 : q == 2 ? 0 : q == 3 ? 4 : 3)) & 31;
    r2 = (leader + (q == 0 ? 2 : q == 1 ? 4 : q == 2 ? 3 : q == 3 ? 3 : 0)) & 31;
    r3 = (leader + (q == 0 ? 3 : q == 1 ? 4 : q == 2 ? 1 : q)) & 31;
  }
  // G == 5 only.  Sums of THREE values over the 5 lanes of a group by reduce-scatter: 3 shuffle
  // stages leave the total of a0 on lane 0, of a1 on lane 1, of a2 on lane 2 (12 additions in 3
  // rounds of <= 5, every lane publishes one value and reads one lane per round) -- against 9
  // stages for three separate all-reduces.  Returns this lane's total (lanes 3, 4: unused).
  //   after stage 1   lane0: u=a0{0,1} v=a1{0}   lane1: u=a2{1} v=a1{1,2}   lane2: u=a2{0,2} v=a0{2}
  //                   lane3: u=a0{3,4} v=a2{3}   lane4: u=a1{3,4} v=a2{4}
  //   after stage 2   lane0: u=a0{0,1,2}  lane1: u=a2{1,4}  lane2: u=a2{0,2,3}  lane3: u=a0{3,4}
  //                   lane4: u=a1{0,3,4}
  //   stage 3         T0 = u0 + u3   T1 = v1 + u4   T2 = u2 + u1
  __device__ __forceinline__ double sum3(double a0, double a1, double a2) const {
    static_assert(G == 5, "sum3 is the 5-lane schedule");
    // lane-constant predicates and plain selects only: no divergent control flow
    const double pub = is0 ? a2 : (is14 ? a0 : a1);
    const double tgt = is03 ? a0 : (is2 ? a2 : a1);
    const double t = tgt + __shfl_sync(kFull, pub, r1);
    const double vo = is0 ? a1 : (is2 ? a0 : a2);
    double u = is1 ? a2 : t;
    const double v = is1 ? t : vo;
    const double x2 = __shfl_sync(kFull, v, r2);
    u += is3 ? 0.0 : x2;
    const double x3 = __shfl_sync(kFull, u, r3);
    return (is1 ? v : u) + x3;
  }
  __device__ __forceinline__ double from_lane(double x, int j) const { return __shfl_sync(kFull, x, lead + j); }
  __device__ __forceinline__ double operator()(double p) const {
    if constexpr (G == 1) {
      return p;
    } else if constexpr (G == 2) {
      return p + __shfl_xor_sync(kFull, p, 1);
    } else if constexpr (G == 4) {
      p += __shfl_xor_sync(kFull, p, 1);
      return p + __shfl_xor_sync(kFull, p, 2);
    } else if constexpr (G == 8) {
      p += __shfl_xor_sync(kFull, p, 1);
      p += __shfl_xor_sync(kFull, p, 2);
      return p + __shfl_xor_sync(kFull, p, 4);
    } else if constexpr (G == 3) {
      const double w2 = p + __shfl_sync(kFull, p, s1);          // lanes q, q+1
      return w2 + __shfl_sync(kFull, p, s2);                    // + q+2
    } else if constexpr (G == 5) {
      const double w2 = p + __shfl_sync(kFull, p, s1);          // q, q+1
      const double w4 = w2 + __shfl_sync(kFull, w2, s2);        // q .. q+3
      return w4 + __shfl_sync(kFull, p, s4);                    // + q+4
    } else if constexpr (G == 6) {
      const double w2 = p + __shfl_sync(kFull, p, s1);
      const double w4 = w2 + __shfl_sync(kFull, w2, s2);
      return w4 + __shfl_sync(kFull, w2, s4);                   // + (q+4, q+5)
    } else {
      static_assert(G == 7, "groups have 1..8 lanes");
      const double w2 = p + __shfl_sync(kFull, p, s1);
      const double w4 = w2 + __shfl_sync(kFull, w2, s2);
      const double w6 = w4 + __shfl_sync(kFull, w2, s4);        // q .. q+5
      return w6 + __shfl_sync(kFull, p, s6);                    // + q+6
    }
  }
};

// RUNS == 6 (5-lane groups only, by-user pass): six runs fill the warp (30 lanes), one rating per
// step -- no cross-group reduction when a level is flushed, a 960-byte contiguous gather.
// RUNS == 2: a warp serves the same piece for a PAIR of runs.  The neighbour rows of the two
// runs are interleaved in memory, so a rating's gather is one contiguous 2*8*NB-byte read
// (fewer L1 wavefronts per byte than two separate rows), and the index loads, the level
// bookkeeping and the cross-group reductions are shared by the two runs.
template <int G, int CH, int UN, int MINB, int RUNS>
__global__ void __launch_bounds__(kWarps * 32, MINB)
segment_pass_kernel(const SegArgs A) {
  constexpr int GR = G * RUNS;                   // lanes per rating
  constexpr int RPS = 32 / GR;                   // ratings per step
  constexpr int SLOTS = UN * RPS;                // ratings per chunk of work (<= 32)
  static_assert(SLOTS <= 32, "a chunk's ids must fit one coalesced 32-lane load");
  extern __shared__ __align__(32) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // one chunk per lane means the row stride is exactly 4*G doubles: a compile-time constant
  const int R = A.R, NBp = (CH == 1) ? 4 * G : A.NBp, RNB = R * NBp;
  const int NCH = NBp >> 2;                      // 32-byte chunks per neighbour row

  constexpr int WB = w_buffers(RUNS);
  double* wbuf = reinterpret_cast<double*>(smem_raw) + (size_t)warp * WB * RUNS * RNB;  // [WB][RUNS][RNB]
  int* ctr = reinterpret_cast<int*>(smem_raw + (size_t)kWarps * WB * RUNS * RNB * 8);
  if (threadIdx.x == 0) *ctr = 0;
  __syncthreads();

  const int grp = lane / GR, lig = lane - grp * GR;
  const int rsel = lig / G, q = lig - rsel * G;  // which run of the group of runs, which lane of the row
  const bool lane_on = grp < RPS;                // lanes past RPS*GR idle (32 % GR of them)
  const int run0 = A.run_base + blockIdx.y * RUNS, run = run0 + rsel;
  // the work schedule (a piece = up to MMSBM_PIECE_LEN ratings of one segment)
  const int32_t* piece_seg = A.sched + 4;
  const int32_t* piece_idx = piece_seg + A.pmax;
  const int32_t* piece_slot = piece_idx + A.pmax;
  const int n_pieces = __ldg(A.sched);
  // A warp starts on piece `first` and claims further ones with an atomic counter: claim t is
  // piece claim_base + t.  With A.counters the counter is global to the launch (one per grid.y),
  // every warp of the grid draws from the same queue, so no CTA is left with a long tail whatever
  // the lengths of the pieces; otherwise the counter is per CTA over its own range of pieces.
  const bool dyn = A.counters != nullptr;
  int* claim = dyn ? A.counters + blockIdx.y : ctr;
  const int seg_lo = dyn ? 0 : blockIdx.x * A.segs_per_cta;
  const int seg_hi = dyn ? n_pieces : min(seg_lo + A.segs_per_cta, n_pieces);
  const int first = dyn ? blockIdx.x * kWarps + warp : seg_lo + warp;
  const int claim_base = dyn ? gridDim.x * kWarps : seg_lo + kWarps;
  // base of this lane's neighbour rows: row(id) = nbr_run + id * RUNS * NBp
  const double* nbr_run = (RUNS == 1) ? A.nbr + (size_t)run * A.nnbr * NBp
                                      : A.nbr + ((size_t)(A.grp_base + blockIdx.y) * A.nnbr * RUNS + rsel) * NBp;
  int coff[CH];                                  // lane-constant chunk offsets (in doubles)
  bool con[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) {
    const int chunk = c * G + q;
    con[c] = lane_on && chunk < NCH;
    coff[c] = con[c] ? 4 * chunk : 0;            // idle lanes re-read chunk 0 (same line)
  }
  const GroupSum<G> group_sum(grp * GR + rsel * G, q);

  // w rows (one per run) of a segment -> shared memory, asynchronously (16-byte pieces)
  auto fetch_w = [&](int s_, int b_) {
#pragma unroll 1
    for (int r2 = 0; r2 < RUNS; ++r2) {
      const double* src = A.wg + ((size_t)(run0 + r2) * A.nseg + s_) * RNB;
      double* dst = wbuf + (size_t)(b_ * RUNS + r2) * RNB;
#pragma unroll 1
      for (int p = lane; p < (RNB >> 1); p += 32) cp_async16(dst + 2 * p, src + 2 * p);
    }
  };

  // prefetched state of a piece: its segment, (piece number, slot) in lanes 0 and 1, and the
  // level boundaries of the segment (lane r <= R holds the start of level r)
  int pi = first, buf = 0;
  int sg = 0, pinfo_pref = 0, bend_pref = 0;
  auto prefetch_piece = [&](int p_, int b_, int& sg_out) {
    MMSBM_DEV_CHECK(p_ >= 0 && p_ < A.pmax);
    sg_out = __ldg(piece_seg + p_);
    MMSBM_DEV_CHECK(sg_out >= 0 && sg_out < A.nseg);
    pinfo_pref = (lane == 0) ? __ldg(piece_idx + p_) : (lane == 1) ? __ldg(piece_slot + p_) : 0;
    if (lane <= R) bend_pref = __ldg(A.seg + (size_t)sg_out * R + lane);
    if constexpr (WB == 2) fetch_w(sg_out, b_);
  };
  if (pi < seg_hi) prefetch_piece(pi, 0, sg);
  cp_async_commit();

  while (pi < seg_hi) {
    const int bend_reg = bend_pref, pinfo = pinfo_pref;
    // claim the next piece, start fetching its descriptors and its w row
    int t = 0;
    if (lane == 0) t = atomicAdd(claim, 1);
    const int pi_next = claim_base + __shfl_sync(kFull, t, 0);
    int sg_next = 0;
    if (pi_next < seg_hi) prefetch_piece(pi_next, buf ^ 1, sg_next);
    cp_async_commit();
    const int slot = __shfl_sync(kFull, pinfo, 1);
    const int beg = __shfl_sync(kFull, bend_reg, 0) + __shfl_sync(kFull, pinfo, 0) * MMSBM_PIECE_LEN;
    const int end = min(beg + MMSBM_PIECE_LEN, __shfl_sync(kFull, bend_reg, R));
    MMSBM_DEV_CHECK(slot >= -1 && slot < A.smax && beg >= 0 && beg <= end);
    // ids of the first chunk; slots past the end read row 0 (in bounds, weight zero)
    int cur_ids = 0;
    if (lane < SLOTS && beg + lane < end) cur_ids = ld_stream(A.adj + beg + lane);
    if constexpr (WB == 2) {
      cp_async_wait<1>();                        // this segment's w has landed
    } else {                                     // single buffer: fetched now (the previous piece is done with it)
      fetch_w(sg, 0);
      cp_async_commit();
      cp_async_wait<0>();
    }
    __syncwarp();
    const double* wb = wbuf + (size_t)((WB == 2 ? buf : 0) * RUNS + rsel) * RNB;
    double* gout = (slot < 0) ? A.wg + ((size_t)run * A.nseg + sg) * RNB
                              : A.partial + ((size_t)run * A.smax + slot) * RNB;

    double4_t g[CH], wr[CH];
    auto flush = [&](int r, bool any) {          // g_r: sum over the groups, then to global
#pragma unroll
      for (int c = 0; c < CH; ++c) {
        double4_t v = g[c];
        if (any) {                               // warp-uniform; an empty level stores zeros
#pragma unroll
          for (int off = 16; off > 0; off >>= 1) {
            if (off < RPS) {
              const double tx = __shfl_down_sync(kFull, v.x, off * GR);
              const double ty = __shfl_down_sync(kFull, v.y, off * GR);
              const double tz = __shfl_down_sync(kFull, v.z, off * GR);
              const double tw = __shfl_down_sync(kFull, v.w, off * GR);
              if (grp + off < RPS) { v.x += tx; v.y += ty; v.z += tz; v.w += tw; }
            }
          }
        }
        if (grp == 0 && con[c]) stg256(gout + r * NBp + coff[c], v);
      }
    };

    // Level-major: the ratings of a segment are stored grouped by level, so the piece is the
    // concatenation of (at most R) level runs.  Each run is cut into chunks of up to SLOTS
    // ratings -- the level, hence w, is warp-uniform inside a chunk; the last chunk of a run is
    // partial (its idle slots gather row 0 with weight zero).
    int lo = beg;                                // start of the part of the piece not yet done
    for (int r = 0; r < R; ++r) {
      const int le = min(end, __shfl_sync(kFull, bend_reg, r + 1));   // end of level r in the piece
#pragma unroll
      for (int c = 0; c < CH; ++c) g[c] = double4_t{0.0, 0.0, 0.0, 0.0};
      const bool any = lo < le;
      if (any) {
#pragma unroll
        for (int c = 0; c < CH; ++c)
          wr[c] = con[c] ? lds32(wb + r * NBp + coff[c]) : double4_t{0.0, 0.0, 0.0, 0.0};
        for (int base = lo; base < le; base += SLOTS) {
          const int cnt = min(SLOTS, le - base); // 1..SLOTS ratings in this chunk
          // NS = steps of this chunk that hold ratings (the tail chunk of a level has fewer)
          auto chunk = [&](auto ns_tag) {
            constexpr int NS = decltype(ns_tag)::value;
            // ---- gather: one 256-bit load per (step, chunk) ----
            double4_t x[NS][CH];
#pragma unroll
            for (int un = 0; un < NS; ++un) {
              const int sl = un * RPS + grp;
              int id = __shfl_sync(kFull, cur_ids, sl & 31);
              if (sl >= cnt) id = 0;             // beyond the chunk: row 0 (in bounds), weight zero
              MMSBM_DEV_CHECK(id >= 0 && id < A.nnbr);
              const double* row = nbr_run + (size_t)id * (RUNS * NBp);
#pragma unroll
              for (int c = 0; c < CH; ++c) x[un][c] = ldg256(row + coff[c]);
            }
            // next chunk's ids (independent of the row loads above); the next chunk starts
            // where this one ends, whatever its level
            {
              const int nxt = base + cnt + lane;
              cur_ids = (lane < SLOTS && nxt < end) ? ld_stream(A.adj + nxt) : 0;
            }
            // all dots first, then the reciprocals, then the accumulation: every row is needed
            // by the first phase, so the loads are issued back to back
            double im[NS];
#pragma unroll
            for (int un = 0; un < NS; ++un) {
              double part = 0.0, part2 = 0.0;
#pragma unroll
              for (int c = 0; c < CH; ++c) {
                part = fma(x[un][c].x, wr[c].x, part); part2 = fma(x[un][c].y, wr[c].y, part2);
                part = fma(x[un][c].z, wr[c].z, part); part2 = fma(x[un][c].w, wr[c].w, part2);
              }
              im[un] = part + part2;
            }
            if constexpr (G == 5 && NS == 3) {
              // one reduce-scatter for the three dots, ONE reciprocal per lane, then the three
              // reciprocals are read back from lanes 0..2 of the group
              const double mine = rcp_clamped(group_sum.sum3(im[0], im[1], im[2]));
#pragma unroll
              for (int un = 0; un < NS; ++un) {
                im[un] = group_sum.from_lane(mine, un);
                if (un * RPS + grp >= cnt) im[un] = 0.0;
              }
            } else {
#pragma unroll
              for (int un = 0; un < NS; ++un) {
                im[un] = rcp_clamped(group_sum(im[un]));
                if (un * RPS + grp >= cnt) im[un] = 0.0;   // idle slot (also the lanes past RPS*GR)
              }
            }
#pragma unroll
            for (int un = 0; un < NS; ++un) {
#pragma unroll
              for (int c = 0; c < CH; ++c) {
                g[c].x = fma(x[un][c].x, im[un], g[c].x); g[c].y = fma(x[un][c].y, im[un], g[c].y);
                g[c].z = fma(x[un][c].z, im[un], g[c].z); g[c].w = fma(x[un][c].w, im[un], g[c].w);
              }
            }
          };
          static_assert(UN <= 6, "extend the step-count dispatch");
          const int ns = (cnt + RPS - 1) / RPS;  // steps that hold ratings, 1..UN (warp-uniform)
          if (ns == UN) chunk(std::integral_constant<int, UN>{});
          else if (ns == 1) chunk(std::integral_constant<int, 1>{});
          else if (UN > 2 && ns == 2) chunk(std::integral_constant<int, (UN > 2 ? 2 : 1)>{});
          else if (UN > 3 && ns == 3) chunk(std::integral_constant<int, (UN > 3 ? 3 : 1)>{});
          else if (UN > 4 && ns == 4) chunk(std::integral_constant<int, (UN > 4 ? 4 : 1)>{});
          else if (UN > 5 && ns == 5) chunk(std::integral_constant<int, (UN > 5 ? 5 : 1)>{});
        }
        lo = le;
      }
      flush(r, any);
    }
    __syncwarp();
    buf ^= 1;
    sg = sg_next;
    pi = pi_next;
  }
  cp_async_wait<0>();
}

// one instantiation unit per CH (seg_inst_ch*.cu) keeps compile time parallel
int launch_segment_pass_ch1(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st);
int launch_segment_pass_pair(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st);
int launch_segment_pass_hexa(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st);
int launch_segment_pass_ch2(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st);
int launch_segment_pass_ch4(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st);
int launch_segment_pass_ch8(const SegArgs& a, int G, int UN, int MINB, dim3 grid, size_t smem, cudaStream_t st);

#define MMSBM_SEG_LAUNCH(Gv, CHv, UNv, MBv) MMSBM_SEG_LAUNCH_R(Gv, CHv, UNv, MBv, 1)
#define MMSBM_SEG_LAUNCH_R(Gv, CHv, UNv, MBv, RUNSv)                                           \
  if (G == Gv && UN == UNv && MINB == MBv) {                                                   \
    auto kern = segment_pass_kernel<Gv, CHv, UNv, MBv, RUNSv>;                                 \
    MMSBM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, dim3(kWarps * 32), smem, st>>>(a);                                            \
    MMSBM_LAUNCH_CHECK("segment_pass_kernel");                                                 \
    return 0;                                                                                  \
  }

}  // namespace mmsbm
