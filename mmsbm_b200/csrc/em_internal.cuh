// Launch helpers of the EM iteration shared by em_step.cu (one GPU) and sharded_run.cu (the
// user-range x item-range sharded loop).  Kernels and their documentation live in em_step.cu.
#pragma once
#include "common.cuh"
#include "segment_pass.cuh"

namespace mmsbm {

constexpr int kPrSlabs = 128;

int env_int(const char* name, int dflt);
int sm_count();                       // multiprocessors of the current device (cached per device)
// resident CTA slots the persistent segment pass leaves free (for NCCL kernels of a sharded run)
void set_reserved_ctas(int n);

// How the S runs of a launch row are served by the segment pass for neighbour rows of NBp
// doubles: runs [0, 6*hexas) six per warp, then `pairs` pairs (pair groups numbered over ALL
// runs, first one = pair_group0), the rest one run per warp from run `single_from`.  A group
// of runs is planned only when its w rows (R levels) fit the shared memory of a CTA: six runs
// fall back to pairs, pairs to one run per warp.  The tables of interleaved rows are filled for
// exactly the planned groups.
struct RunPlan { int hexas, pairs, pair_group0, single_from; };
RunPlan plan_runs(int NBp, int R, int n_runs, bool hexa_table);

int launch_prep_p(const double* pr, int K, int L, int R, int ldk, int ldl, int n_runs, double* pw_u,
                  double* pn_u, double* pw_i, double* pn_i, cudaStream_t st);

// dst[(grp*n_dst + row0 + id)*gs + j][ld] <- src[(gs*grp + j)*n_src + id][ld] for grp in
// [group0, group0+groups), id < n_src: the rows of run groups side by side, written into a table
// of n_dst rows per group starting at row row0 (gs == 1: a plain copy of run `grp`)
int launch_interleave(const double* src, double* dst, int n_src, int n_dst, int row0, int ld,
                      int group0, int groups, int gs, cudaStream_t st);

int launch_w(const double* own, const double* pw, double* W, int M, int LD, int RNB, int n_runs,
             cudaStream_t st);
// Where launch_n ALSO writes the new rows (row_n_kernel stores them itself, the tiled path copies them
// afterwards), in the run-interleaved layout of a gather table that
// spans all ranks (a sharded run publishes its new rows this way instead of re-reading them with
// interleave_runs_kernel): table t serves the runs [gs*group0, gs*(group0+groups)) and holds
// dst[((run/gs) * n_all + row0 + row) * gs + run%gs][ld].
struct RowPublish {
  double* dst[3];
  int gs[3], group0[3], groups[3];
  int n_all, row0;
};
int launch_n(const double* G, const double* pn, const double* own, const int32_t* deg, double* out,
             int M, int LD, int RNB, int normalize, int n_runs, cudaStream_t st,
             const RowPublish* publish = nullptr);

int launch_segment_pass_and_fixup(SegArgs a, const double* nbr_pairs, const double* nbr_hexa,
                                  int64_t n_ratings, int n_runs, cudaStream_t st, bool no_long_segments = false);

// n_pr from the side whose segments carry the accumulation: Acc = sum_seg own (x) g over `nseg`
// segments (kPrSlabs partial sums, fixed order), x P, optionally normalised over the rating axis
int launch_pr(const double* own, const double* g, double* partial, const double* pr, double* pr_out,
              int nseg, int NA, int lda, int NBp, int K, int L, int R, int n_runs, bool transposed,
              bool normalize, cudaStream_t st);
int launch_finalize_pr(double* pr, int kl_total, int R, cudaStream_t st);

// em_small.cu: a whole fit of a small one-run problem in one cooperative launch.  Returns
// MMSBM_ERANGE when the shape (or the device, or MMSBM_COOP=0) is not served: take the other path.
// long_segments: whether a schedule holds a segment cut into pieces (0/1) when the caller has read
// the schedule headers, -1 to have them read here (one stream synchronisation).
bool em_small_applicable(int64_t N, int R, int K, int L, int S);
size_t em_small_partial_elems(int R, int K);
int launch_em_small(const int32_t* useg, const int32_t* uadj, const int32_t* udeg, const int32_t* iseg,
                    const int32_t* iadj, const int32_t* ideg, const int32_t* usched, const int32_t* isched, int64_t N,
                    int U, int I, int R, int K, int L, int S, int iterations, double* theta_a, double* eta_a,
                    double* pr_a, double* theta_b, double* eta_b, double* pr_b, double* partial, size_t partial_elems,
                    cudaStream_t st, int long_segments = -1);

// reductions.cu: observed-data log-likelihood of S runs (mmsbm_loglik without the argument checks)
int launch_loglik(const int32_t* useg, const int32_t* uadj, const int32_t* usched, int64_t N, int U, int I,
                  int R, int K, int L, int S, const double* theta, const double* eta, const double* pr,
                  double* out, void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace mmsbm
