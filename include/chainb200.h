/*
 * chainb200.h -- C ABI of libchainb200.so, the B200 (sm_100a) engine for the hot path of
 * ChainPartitioners.jl: the partition cost oracle over sparse column ranges and the
 * split-point searches that consume it.
 *
 * The reference is pure Julia with no FFI of its own; every entry point below names the Julia
 * method(s) it replaces (paths relative to the reference's src/).  The Julia-side binding a
 * maintainer would add is julia/ChainPartitionersB200.jl (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / CUDA types in any signature;
 *   - all indices are 1-based Int64 exactly as Julia stores SparseMatrixCSC.colptr / .rowval and
 *     SplitPartition.spl; rows must be sorted and unique within a column (the SparseMatrixCSC
 *     invariant);
 *   - "host" pointers may be pageable or pinned; *_device variants take device pointers;
 *   - every function returns 0 on success, <0 on error (cpb_last_error() gives the message);
 *     nothing throws across the boundary;
 *   - handles own device memory only; host arrays are never retained after a call returns;
 *   - one CUDA stream per library instance; calls are serialised; there is NO CPU fallback: every
 *     compute entry point fails with CPB_ERR_CUDA when no device is usable.
 *
 * Lifetimes
 *   - a cpb_matrix must outlive every cpb_oracle / cpb_prefix created from it (the oracle reads the
 *     matrix's device arrays; destroy oracles first).  Handles belong to the device that was current
 *     when they were created: cpb_init(other_device) releases the library's cached blocks and
 *     recreates the stream, and handles of the old device must not be used (or destroyed) after it.
 *
 * Streams
 *   - entry points that take HOST arrays return when their results are in those arrays.
 *   - entry points that take or fill DEVICE arrays (cpb_matrix_create_device,
 *     cpb_oracle_query_device) ENQUEUE work on the library's own non-blocking stream and may
 *     return before it has run: arrays produced on another stream (torch's, the caller's) must be
 *     complete before the call, and cpb_synchronize() must return before another stream reads
 *     what the call wrote.
 */
#ifndef CHAINB200_H
#define CHAINB200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define CPB_OK 0
#define CPB_ERR_ARG (-1)         /* invalid argument */
#define CPB_ERR_UNSUPPORTED (-2) /* model/method combination the reference has no method for, or not built yet */
#define CPB_ERR_CUDA (-3)        /* CUDA runtime error / no device */
#define CPB_ERR_INFEASIBLE (-4)  /* width constraint cannot be met (reference: @assert j0 < j', DynamicChunker.jl:39) */

/* ---- cost models ------------------------------------------------------------------------- */
enum {
  CPB_MODEL_WORK = 0,         /* AffineWorkModel                          WorkCosts.jl:5-17 */
  CPB_MODEL_CONNECTIVITY = 1, /* AffineConnectivityModel                  ConnectivityCosts.jl:7-20 */
  CPB_MODEL_MONOSYM = 2,      /* AffineMonotonizedSymmetricConnectivityModel  MonotonizedSymmetricConnectivityCosts.jl:5-33 */
  CPB_MODEL_SYMCONN = 3,      /* AffineSymmetricConnectivityModel         SymmetricConnectivityCosts.jl:5-19 */
  CPB_MODEL_HYPEREDGE = 4,    /* AffineHyperedgeCutModel                  HyperedgeCutCosts.jl:7-21 */
  CPB_MODEL_SYMEDGECUT = 5,   /* AffineSymmetricEdgeCutModel              SymmetricEdgeCutCosts.jl:5-18 */
  CPB_MODEL_ENVELOPE = 6,     /* AffineEnvelopeModel                      EnvelopeCosts.jl:5-20 */
  CPB_MODEL_COLBLOCK = 7,     /* ColumnBlockComponentCostModel            BlockCosts.jl:1-17 */
  CPB_MODEL_BLOCK = 8,        /* BlockComponentCostModel                  BlockCosts.jl:19-44 */
  CPB_MODEL_SECCONN = 10,           /* AffineSecondaryConnectivityModel with a row partition Pi: the cost of row part k as a function of the column
                                       range [i, i') that is local to it (decreasing)   SecondaryConnectivityCosts.jl:5-102 */
  CPB_MODEL_PRIMEDGE = 11,          /* AffinePrimaryEdgeCutModel(a, b_v, b_self_pin, b_cut_pin) with Pi      PrimaryEdgeCutCosts.jl:5-66 */
  CPB_MODEL_SECEDGE = 12,           /* AffineSecondaryEdgeCutModel(a, b_v, b_self_pin, b_cut_pin) with Pi    SecondaryEdgeCutCosts.jl:5-97 */
  CPB_MODEL_PRIMCONN = 9            /* AffinePrimaryConnectivityModel(a, b_v, b_p, b_local, b_remote) with a row partition Pi: a net of part k's
                                       columns is local if row part k owns it   PrimaryConnectivityCosts.jl:5-86, PartwiseCounts.jl:1-101 */
};

/* coef[] by kind, evaluated left to right without FMA contraction (e.g. ConnectivityCosts.jl:20):
 *   WORK                 alpha, beta_vertex, beta_pin
 *   CONNECTIVITY/ENVELOPE alpha, beta_vertex, beta_pin, beta_net
 *   MONOSYM              alpha, beta_vertex, beta_over_pin, beta_dia_net, delta_pins
 *   SYMCONN              alpha, beta_vertex, beta_pin, beta_local_net, beta_remote_net
 *   HYPEREDGE            alpha, beta_vertex, beta_pin, beta_self_net, beta_cut_net
 *   SYMEDGECUT           alpha, beta_vertex, beta_self_pin, beta_cut_pin
 * is_float = 0: Int64 coefficients and costs (coef[] integer valued, |cost| < 2^53);
 * is_float = 1: Float64.
 * COLBLOCK / BLOCK: block_component(f, w) (BlockCosts.jl:41-44) tabulated by the caller, because
 * Julia functors cannot cross the ABI:
 *   alpha_col[w], w = 0..w_tab;  beta_col[r*(w_tab+1) + w], r = 0..R-1 (COLBLOCK: R = 1);
 *   beta_row[r*(u_tab+1) + u], u = 0..u_tab (BLOCK only; u = size of a row part).
 * COLBLOCK parts wider than w_tab columns have no tabulated cost: cpb_oracle_query returns +Inf for
 * them (the table is normally shrunk to the widest part a ConstrainedCost allows, so such a part is
 * infeasible anyway); the solvers never evaluate them. */
typedef struct cpb_model {
  int32_t kind;
  int32_t is_float;
  double coef[8];
  int32_t R;
  int32_t w_tab;
  int32_t u_tab;
  int32_t _pad;
  const double* alpha_col;
  const double* beta_col;
  const double* beta_row;
} cpb_model;

/* ConstrainedCost(f, w, w_max) (Costs.jl:105-147): w(j,j') = w_coef[0] + (j'-j) w_coef[1] +
 * (colptr[j']-colptr[j]) w_coef[2]; VertexCount() = {0,1,0} (SparseColorArrays.jl:1-6).
 * enabled = 0: FeasibleCost (Costs.jl:164-171). */
typedef struct cpb_constraint {
  int32_t enabled;
  int32_t _pad;
  int64_t w_coef[3];
  int64_t w_max;
} cpb_constraint;

/* ---- library ----------------------------------------------------------------------------- */
const char* cpb_last_error(void);
int cpb_version(void);
/* Selects the CUDA device for this process (one process per GPU). Returns CPB_ERR_CUDA if none. */
int cpb_init(int device);
int cpb_device_count(void);
/* Blocks until all queued work of the library stream has finished. */
int cpb_synchronize(void);
/* Returns the device memory the library keeps cached between calls (its free list of large blocks and the stream-ordered
 * pool) to the driver.  Handles stay valid. */
int cpb_trim_memory(void);

/* ---- matrices ---------------------------------------------------------------------------- */
typedef struct cpb_matrix cpb_matrix;
/* Copies a SparseMatrixCSC pattern (A.colptr, A.rowval) to the device (32-bit, 0-based there). */
int cpb_matrix_create(int64_t m, int64_t n, int64_t nnz, const int64_t* colptr, const int64_t* rowval, cpb_matrix** out);
/* The same for a SparseMatrixCSC{Tv, Int32} (the reference is generic in the index type Ti; half the upload). */
int cpb_matrix_create_i32(int64_t m, int64_t n, int64_t nnz, const int32_t* colptr, const int32_t* rowval, cpb_matrix** out);
/* Same from device-resident Int64 arrays (inputs already in HBM). */
int cpb_matrix_create_device(int64_t m, int64_t n, int64_t nnz, const int64_t* d_colptr, const int64_t* d_rowval, cpb_matrix** out);
int cpb_matrix_dims(const cpb_matrix* A, int64_t* m, int64_t* n, int64_t* nnz);
/* Copies the pattern back as 1-based Int64 host arrays (colptr: n+1, rowval: nnz). */
int cpb_matrix_get(const cpb_matrix* A, int64_t* colptr_out, int64_t* rowval_out);
void cpb_matrix_destroy(cpb_matrix* A);
/* adjointpattern(A) (util.jl:67-95): CSC pattern of the transpose, built on the device. */
int cpb_adjointpattern(cpb_matrix* A, cpb_matrix** out);

/* A[:, col_prm] with row r renamed row_new[r] -- the first step of compute_objective for non-contiguous partitions
 * (Costs.jl:34-39, 52-57: A_prm = A[:, Phi_dom.prm]; PrimaryConnectivityCosts.jl:88-163, WorkCosts.jl:63-81,
 * EnvelopeCosts.jl:100-129).  col_prm: n entries, row_new: m entries, both 1-based permutations; NULL = identity.
 * A MapPartition of the rows becomes a SplitPartition by renaming the rows part by part. */
int cpb_matrix_permute(cpb_matrix* A, const int64_t* col_prm, const int64_t* row_new, cpb_matrix** out);

/* ---- 2-D prefix structures (SparsePrefixMatrices.jl) ---------------------------------------- */
typedef struct cpb_prefix cpb_prefix;
/* dominancecount!(hint, m, n, N, pos, idx) / dominancesum!(hint, m, n, N, pos, idx, val) (SparsePrefixMatrices.jl:33-58,
 * 440-460) and rookcount!(hint, N, idx) / rooksum!(hint, N, idx, val) (:840-851, 1056-1063).  pos (n+1) and idx (N) are the
 * 1-based Int64 arrays Julia holds; pos == NULL selects the rook form (point q sits in column q, n == N, m == N);
 * val == NULL builds counts only.  Values are 64-bit integers, sums wrap like Julia's Int64 / UInt64.  The hint and the
 * b / H / b' layout arguments of the reference have no device counterpart: one wavelet-matrix index serves all of them. */
int cpb_prefix_create(int64_t m, int64_t n, int64_t N, const int64_t* pos, const int64_t* idx, const int64_t* val, cpb_prefix** out);
/* C[i, j] = #{points (r, c): r <= i-1, c <= j-1} and S[i, j] = the sum of their values, 1 <= i <= m+1, 1 <= j <= n+1
 * (getindex, SparsePrefixMatrices.jl:187-254, 537-604, 660-689, 957-1021, 1137-1206, 1246-1273).  Either output may be NULL. */
int cpb_prefix_query(cpb_prefix* P, int64_t Q, const int64_t* i, const int64_t* j, int64_t* count_out, int64_t* sum_out);
void cpb_prefix_destroy(cpb_prefix* P);

/* ---- cost oracles ------------------------------------------------------------------------ */
typedef struct cpb_oracle cpb_oracle;
/* oracle_stripe(hint, mdl, A[, Pi]) (Costs.jl:3-7, ConnectivityCosts.jl:47-56, Monotonized...:77-92,
 * SymmetricConnectivityCosts.jl:29-45, HyperedgeCutCosts.jl:32-42, SymmetricEdgeCutCosts.jl:28-35,
 * EnvelopeCosts.jl:56-64, BlockCosts.jl:58-64).  Builds the link arrays (SparseColorArrays.jl:72-118,
 * 177-229, 281-318) and the 2-D dominance index (replacing SparsePrefixMatrices.jl:462-534 / 610-655 /
 * 695-702: one wavelet-matrix index serves every hint).  pi_spl/pi_K: row SplitPartition for BLOCK. */
int cpb_oracle_create(cpb_matrix* A, const cpb_model* mdl, const int64_t* pi_spl, int64_t pi_K, cpb_oracle** out);
void cpb_oracle_destroy(cpb_oracle* f);
/* ocl(j, j', k) for Q queries (ConnectivityCosts.jl:58-64 etc.).  k may be NULL.  Costs are returned
 * as Float64 (exact for Int64 models below 2^53). */
int cpb_oracle_query(cpb_oracle* f, int64_t Q, const int64_t* j, const int64_t* jp, const int64_t* k, double* cost_out);
int cpb_oracle_query_device(cpb_oracle* f, int64_t Q, const int64_t* d_j, const int64_t* d_jp, double* d_cost_out);
/* Raw counts: which = 0 pincount, 1 netcount, 2 dianetcount, 3 selfnetcount, 4 selfpincount
 * (SparseColorArrays.jl:9-43, 47-152, 72-99, 156-256, 260-345); builds the structure on first use. */
int cpb_count_query(cpb_matrix* A, int which, int64_t Q, const int64_t* j, const int64_t* jp, int64_t* out);
/* bound_stripe(A, K, mdl-or-ocl) ./ 1 (WorkCosts.jl:37-51, ConnectivityCosts.jl:22-35,
 * MonotonizedSymmetricConnectivityCosts.jl:35-66,94-105, EnvelopeCosts.jl:30-54). */
int cpb_bound_stripe(cpb_oracle* f, int64_t K, double out[2]);
/* bottleneck_value / total_value of a SplitPartition (Costs.jl:26-66). */
int cpb_objective(cpb_oracle* f, int total, int64_t K, const int64_t* spl, double* out);

/* ---- partition_stripe -------------------------------------------------------------------- */
enum {
  CPB_SPLIT_DYNAMIC_BOTTLENECK = 0, /* partition_stripe(A, K, DynamicBottleneckSplitter(f))  DynamicSplitter.jl:15-50 */
  CPB_SPLIT_DYNAMIC_TOTAL = 1,      /* partition_stripe(A, K, DynamicTotalSplitter(f))       DynamicSplitter.jl:15-50 */
  CPB_SPLIT_BISECT_COST = 2,        /* BisectCostBottleneckSplitter(f, eps)      BisectCostBottleneckSplitter.jl:6-63 */
  CPB_SPLIT_LAZY_BISECT_COST = 3,   /* LazyBisectCostBottleneckSplitter(f, eps)  LazyBisectCostBottleneckSplitter.jl:8-70,140-258,260-388 */
  CPB_SPLIT_EQUI = 5,               /* EquiSplitter()                            EquiPartitioner.jl:3-9 */
  CPB_SPLIT_CONVEX_TOTAL = 8,       /* partition_stripe(A, K, ConvexTotalSplitter(f))  ConvexTotalChunker.jl:26-55 (quadrangle-inequality models) */
  CPB_SPLIT_CONCAVE_TOTAL = 9,      /* partition_stripe(A, K, ConcaveTotalSplitter(f))  ConcaveTotalChunker.jl:26-55, 143-181 (sequential queue routine, one device thread) */
  /* partition_stripe(A, K, ::AbstractDynamicChunker) DynamicSplitter.jl:52-87,249-314: the same K-part recurrence
     and `<=` tie rule as the splitter form with the part index as the inner loop -> identical split vectors */
  CPB_SPLIT_DYNAMIC_BOTTLENECK_CHUNKER = 10, /* partition_stripe(A, K, DynamicBottleneckChunker(f)) */
  CPB_SPLIT_DYNAMIC_TOTAL_CHUNKER = 11,      /* partition_stripe(A, K, DynamicTotalChunker(f)) */
  CPB_SPLIT_BISECT_INDEX = 12,               /* BisectIndexBottleneckSplitter(f): exact bottleneck   BisectIndexBottleneckSplitter.jl:5-81 */
  /* the Flip family: costs that DEcrease as the part grows (the secondary models) */
  CPB_SPLIT_FLIP_BISECT_COST = 6,            /* FlipBisectCostBottleneckSplitter(f, eps)       BisectCostBottleneckSplitter.jl:70-127 */
  CPB_SPLIT_LAZY_FLIP_BISECT_COST = 7,       /* LazyFlipBisectCostBottleneckSplitter(f, eps)   LazyBisectCostBottleneckSplitter.jl:79-138 */
  CPB_SPLIT_FLIP_BISECT_INDEX = 13           /* FlipBisectIndexBottleneckSplitter(f)           BisectIndexBottleneckSplitter.jl:87-166 */
};
/* -> spl_out[K+1] (SplitPartition{Int64}(K, spl), Partitions.jl:3-6); con may be NULL. */
int cpb_partition_stripe(cpb_oracle* f, int method, const cpb_constraint* con, double eps, int64_t K, int64_t* spl_out);
/* B independent partition_stripe problems in one launch, one cluster each.  Every result is identical to
 * cpb_partition_stripe(f[b], method[b], NULL, eps[b], K[b], spl_out[b]).  Methods: CPB_SPLIT_BISECT_INDEX,
 * CPB_SPLIT_FLIP_BISECT_COST, CPB_SPLIT_LAZY_FLIP_BISECT_COST, CPB_SPLIT_FLIP_BISECT_INDEX (else CPB_ERR_UNSUPPORTED).
 * Oracles may repeat and may belong to different matrices of this device; eps may be NULL when no Flip-cost method is
 * present; spl_out[b] holds K[b] + 1 entries.  Any invalid problem fails the whole call before any launch (the message
 * names the problem) and no spl_out is written.  B = 0 returns CPB_OK; a batch does not update cpb_bisect_stats. */
int cpb_partition_stripe_batch(int64_t B, cpb_oracle* const* f, const int* method, const double* eps, const int64_t* K,
                               int64_t* const* spl_out);
/* Clusters of the batch kernel the device keeps resident at once (cudaOccupancyMaxActiveClusters): larger batches queue. */
int cpb_partition_stripe_batch_capacity(int* clusters_out);

/* partition_stripe(A, K, method(ConstrainedCost(f, w, w_max))) with the weight given as a cost model of its own
 * (Costs.jl:105-147: the reference turns w into an oracle and tests w(j, j') > w_max for the windows of every constrained
 * solver, column_constraints DynamicSplitter.jl:144-173).  w is a cpb_oracle created by cpb_oracle_create over the SAME
 * cpb_matrix as f (else CPB_ERR_ARG); w(j, j') is its Int64 cost of columns j..j'-1.  Accepted weights: integer
 * AffineWorkModel, AffineConnectivityModel and AffineMonotonizedSymmetricConnectivityModel (square A) with
 * beta_vertex, beta_pin / beta_over_pin, beta_net / beta_dia_net >= 0 (delta_pins is free) -- they cannot shrink when the
 * range grows, so the windows are monotone.  An AffineWorkModel weight takes the cpb_constraint path.  Float64 weights,
 * negative betas and every other model return CPB_ERR_UNSUPPORTED, as do the Bisect, Flip and Equi methods.  Methods:
 * CPB_SPLIT_DYNAMIC_BOTTLENECK / _TOTAL (and their _CHUNKER forms), CPB_SPLIT_CONVEX_TOTAL, CPB_SPLIT_CONCAVE_TOTAL.
 * w_max below w(j, j) makes every part infeasible; an infeasible chain returns [1, 1, ..., 1, n+1]. */
int cpb_partition_stripe_weighted(cpb_oracle* f, int method, cpb_oracle* w, int64_t w_max, double eps, int64_t K, int64_t* spl_out);
/* The windows of such a weight, 1-based, n + 1 entries each (index c - 1 holds column c = 1..n+1):
 *   first_fit_out[j' - 1] = the smallest j in [1, j'] with j == j' or w(j, j') <= w_max,
 *   reach_out[j - 1]      = the largest j' in [j, n+1] with j' == j or w(j, j') <= w_max.
 * Builds w's dominance index on first use (a second wavelet index when f and w are different oracles). */
int cpb_weight_windows(cpb_oracle* w, int64_t w_max, int64_t* first_fit_out, int64_t* reach_out);

/* The speculation plan of one round, as a pure host computation (no device needed): the `nodes` nodes (heap indices in
 * the bisection tree, root = 0, left child 2i+1 = "probe i was feasible"; -1 = unused slot) that are probed concurrently
 * when the bracket is (c_lo, c_hi], the initial bracket was (c_lo0, c_hi0] and `upper_bound` (0 = unknown) bounds the
 * optimum from above.  The set always contains the root and is closed under taking parents; which nodes are in it never
 * changes the result, only how many rounds the bisection needs. */
int cpb_bisect_plan(double c_lo, double c_hi, double eps, int nodes, double c_lo0, double c_hi0, double upper_bound, int32_t* ids_out);
/* Host-only: the leading probes of the loop BisectCostBottleneckSplitter.jl:41-60 that an upper bound on the optimal bottleneck
 * settles without running them (every threshold >= upper_bound (1 + eps)^2 is feasible and cannot be the last feasible probe --
 * unless it is the probe that ends the loop, which is left to run).  Returns the c_hi they leave and their number. */
int cpb_bisect_prewalk(double c_lo, double c_hi, double eps, double upper_bound, double* c_hi_out, int32_t* probes_out);
/* Diagnostics of the most recently finished bisection of this process: out[0] = rounds (batches of concurrent
 * probes), out[1] = probes the sequential loop of the reference would have run, out[2] = thresholds probed
 * speculatively in total, out[3] = initial c_lo, out[4] = initial c_hi, out[5] = the planner's upper bound (0 = none), out[6] = final c_lo,
 * out[7] = final c_hi. */
int cpb_bisect_stats(double out[8]);

/* ---- one stripe solve over several GPUs (one process per GPU) ----------------------------------
 * The reference has no counterpart (it is single-threaded); these entry points stand where a maintainer would put a
 * `Distributed`/MPI.jl driver around partition_stripe(A, K, LazyBisectCostBottleneckSplitter(...)) (LazyBisectCost...:140-258).
 * The communicator is owned by the library (NCCL, loaded at run time): rank 0 obtains the 128-byte id with
 * cpb_comm_unique_id, ships it to the other ranks by any means (MPI.jl bcast, a file, torch.distributed), and every rank
 * calls cpb_comm_init after cpb_init(its device).  All sharded calls are COLLECTIVE: every rank makes the same call with
 * the same matrix, model, K and eps.
 *
 * cpb_sharded_matrix_create: every rank passes the complete colptr; of rowval only the rank's block of CSC positions
 * [q_lo, q_hi) (cpb_shard_range) is read and uploaded -- pass the whole array (rowval_is_block = 0) or just the block
 * (rowval_is_block = 1, rowval[0] = entry q_lo).
 * cpb_partition_stripe_sharded: BisectCost / LazyBisectCost with the AffineConnectivityModel or the
 * AffineMonotonizedSymmetricConnectivityModel (square A).  Link construction by blocks of CSC positions: local stable sort
 * by row, the per-row "last position" array (m x 4 bytes) carried down the ranks once (ncclSend/Recv), one in-place
 * all-gather of the link shards (nnz x 4 bytes); bisection rounds of world x 15 thresholds, rank r probing its 15, one
 * all-gather of the per-threshold results per round.  Every rank returns the same split vector -- the single-GPU (and the
 * reference's) one.  The monotonized symmetric model streams the links of A + I: the ranks combine their "diagonal present"
 * flags (one n-byte MAX all-reduce), every rank's block becomes [img(q_lo), img(q_hi)) of A + I positions (a virtual diagonal
 * goes with the last element of its column, rank 0 starts at 0), and one in-place broadcast per rank gathers the blocks.
 * cpb_partition_stripe_sharded_emulated plays `world` ranks one after the other on this GPU (tests; no NCCL).
 * cpb_sharded_adjointpattern: adjointpattern (util.jl:67-95) of a sharded matrix, collective; the result holds the complete
 * colptr of the transpose and this rank's block of its rowval (the same cpb_shard_range blocks: nnz is unchanged).  Row
 * histograms of the blocks are all-gathered (m x 4 bytes per rank), each entry is routed to the rank owning its position in
 * the transpose with grouped ncclSend/Recv (8 bytes per nonzero).  Rectangular patterns are fine.
 * cpb_adjointpattern_sharded_emulated: the same construction with `world` ranks played on this GPU, assembled into one
 * whole matrix (tests).
 * cpb_sharded_matrix_get: the 1-based colptr (n + 1 entries) and this rank's block of rowval (q_hi - q_lo entries, 1-based),
 * and the 0-based half-open block [q_lo, q_hi) of CSC positions; any output may be NULL.
 * cpb_sharded_stats: out[0] = world, [1] = host ms until the construction was queued, [2] = ms of the bisection (incl.
 * waiting for the construction), [3] = bisection rounds, [4] = link gather bytes (of A + I for the monotonized symmetric
 * model), [5] = carry bytes per hop, [6] = threshold all-gather bytes, [7] = thresholds per round, [8] = bytes of transpose
 * pairs this rank received from other ranks in its last cpb_sharded_adjointpattern, [9] = its histogram all-gather bytes. */
typedef struct cpb_sharded cpb_sharded;
int cpb_comm_unique_id(char id_out[128]);
int cpb_comm_init(const char id[128], int rank, int world);
int cpb_comm_destroy(void);
int cpb_comm_info(int* rank, int* world);
int cpb_shard_range(int64_t nnz, int rank, int world, int64_t* q_lo, int64_t* q_hi);
int cpb_sharded_matrix_create(int64_t m, int64_t n, int64_t nnz, const int64_t* colptr, const int64_t* rowval, int rowval_is_block,
                              cpb_sharded** out);
void cpb_sharded_matrix_destroy(cpb_sharded* A);
int cpb_partition_stripe_sharded(cpb_sharded* A, const cpb_model* mdl, int method, double eps, int64_t K, int64_t* spl_out);
int cpb_partition_stripe_sharded_emulated(cpb_matrix* A, const cpb_model* mdl, int method, double eps, int64_t K, int world,
                                          int64_t* spl_out);
int cpb_sharded_adjointpattern(cpb_sharded* A, cpb_sharded** out);
int cpb_adjointpattern_sharded_emulated(cpb_matrix* A, int world, cpb_matrix** out);
int cpb_sharded_matrix_get(const cpb_sharded* A, int64_t* colptr_out, int64_t* rowval_block_out, int64_t* q_lo, int64_t* q_hi);
int cpb_sharded_stats(double out[16]);

/* ---- pack_stripe ------------------------------------------------------------------------- */
enum {
  CPB_PACK_DYNAMIC_TOTAL = 0, /* pack_stripe(A, DynamicTotalChunker(ConstrainedCost(f, w, w_max))[, Pi])  DynamicChunker.jl:20-56 */
  CPB_PACK_CONVEX_TOTAL = 1,  /* pack_stripe(A, ConvexTotalChunker(ConstrainedCost(...)))                 ConvexTotalChunker.jl:141-265 */
  CPB_PACK_CONCAVE_TOTAL = 2, /* ConcaveTotalChunker.jl:9-114 */
  CPB_PACK_OVERLAP = 3,       /* pack_stripe(A, OverlapChunker(rho, w_max))                               OverlapChunker.jl:6-75 */
  CPB_PACK_STRICT = 4,        /* pack_stripe(A, StrictChunker(w_max))                                     StrictChunker.jl:5-54 */
  CPB_PACK_EQUI = 5           /* pack_stripe(A, EquiChunker(w))                                           EquiPartitioner.jl:15-21 */
};
/* f may be NULL for OVERLAP / STRICT / EQUI (A is used).  spl_out must hold n+1 entries; K_out
 * receives the number of chunks; n_nets_out (n entries or NULL) receives OverlapChunker's n_nets. */
int cpb_pack_stripe(cpb_matrix* A, cpb_oracle* f, int method, const cpb_constraint* con, double rho, int64_t w_max,
                    int64_t* spl_out, int64_t* K_out, int64_t* n_nets_out);

/* ---- measurement hooks (bench.py) -------------------------------------------------------- */
/* When enabled, phases are bracketed with CUDA events on the library stream. */
int cpb_profile_enable(int on);
int cpb_profile_reset(void);
/* Copies up to cap entries: names (char[32] each), total milliseconds, launches, algorithmic bytes. */
int cpb_profile_get(int cap, char* names, double* ms, int64_t* launches, double* bytes);
/* Number of kernels launched by the library since cpb_profile_reset(). */
int64_t cpb_launch_count(void);
/* Device-side stopwatch: records a CUDA event on the library stream / records a second one, waits
 * for it and returns the elapsed milliseconds between the two. */
int cpb_timer_start(void);
int cpb_timer_stop(double* ms_out);

#ifdef __cplusplus
}
#endif
#endif
