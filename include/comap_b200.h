/*
 * comap_b200.h -- C ABI of libcomap_b200.so: CoMap's data-parallel hot path on B200.
 *
 * The reference (jydu/comap 1.6.0a) has no plugin / FFI interface: its hot path is four
 * C++ call sites into Bio++ objects (SURVEY.md s8b).  Each entry point below replaces one
 * of those call sites; the citation names the reference file:line (relative to
 * /root/reference) whose semantics it keeps.  A C++ front-end that mirrors CoMap.cpp's
 * flow on top of this ABI is comap_b200/host/ (binary `comap_b200`); INTEGRATION.md shows
 * the stub a CoMap maintainer would add to call it from CoETools.cpp.
 *
 * Conventions
 *   - Every function returns 0 on success, non-zero on error; cmb_last_error() gives the
 *     message (maps onto the reference's bpp::Exception -> message -> exit(-1),
 *     CoMap.cpp:730-734).  There is NO CPU fallback: without a CUDA device
 *     cmb_ctx_create fails.
 *   - All pointers are caller-allocated HOST buffers (pinned memory makes copies faster;
 *     cmb_host_alloc provides it) unless the name ends in _dev.  Any output pointer
 *     documented "nullable" may be NULL.
 *   - A cmb_ctx is bound to one GPU and one CUDA stream; it is not thread-safe.  Multi-GPU
 *     runs use one context per GPU (one process each, or one thread each in one process),
 *     shard work with the shard_* arguments and exchange the null samples with NCCL through
 *     cmb_comm_* / cmb_null_intra_sharded (or, with the caller's own plumbing, the *_dev
 *     entry points).
 *   - tree  : n_nodes nodes, ids in Newick post-order (children before parent), root =
 *             n_nodes-1 with parent -1.  Branch b = edge above node b, B = n_nodes-1.
 *             Leaf k (k-th childless node in id order) is row k of every alignment.
 *             Lengths below 1e-6 are raised to 1e-6 as Bio++ does.
 *   - model : A states (2..32), generator Q row-major A*A, reversible w.r.t. pi and
 *             normalised by the caller; C rate classes (1..32).
 *   - sites : uint8 codes, tip-major [T][S]; code_mask[code] = bitmask of compatible
 *             states, so ambiguity codes are multi-state tips, not gaps.
 *   - Substitution register: Total (one type), optionally weighted (weight_xy).
 */
#ifndef COMAP_B200_H
#define COMAP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cmb_ctx cmb_ctx;

/* nijt= : PhylogeneticsApplicationTools::getSubstitutionCount, CoMap.cpp:152 */
enum { CMB_COUNT_UNIFORMIZATION = 0, CMB_COUNT_DECOMPOSITION = 1, CMB_COUNT_NAIVE = 2,
       CMB_COUNT_LAPLACE = 3 /* Laplace(trunc=10): unweighted; pinned by Myo_laplace.vec */,
       CMB_COUNT_LABEL = 4 /* Label: substitution x -> y counts as its label 1..A(A-1) (for MI, CoETools.cpp:577-589) */,
       CMB_COUNT_ONE_JUMP = 5 /* ProbOneJump: probability of at least one substitution on the branch given its ends */ };
/* nijt=Laplace(trunc=k), k in 2..20: the truncation order rides in the upper bits of count_method */
#define CMB_COUNT_LAPLACE_TRUNC(k) (CMB_COUNT_LAPLACE | ((k) << 8))
/* statistic= : CoETools::getStatistic, CoETools.cpp:535-600; Statistics.h:164-295 */
enum {
  CMB_STAT_CORRELATION = 0,
  CMB_STAT_COVARIANCE = 1,
  CMB_STAT_COSINUS = 2,
  CMB_STAT_COSUBSTITUTION = 3,
  CMB_STAT_COMPENSATION = 4,
  CMB_STAT_CORRECTED_CORRELATION = 5, /* Statistics.h:176-205; mean vector as CoMap.cpp:350-359 */
  CMB_STAT_MI = 6, /* MI(threshold=..) without nijt=Label: DiscreteMutualInformationStatistic over the
                     bounds {0, threshold, 10000} (CoETools.cpp:590-595, Statistics.h:307-329) */
  CMB_STAT_MI_LABEL = 7 /* MI with nijt=Label and nijt.average=no: one category per substitution label, bounds
                           -0.5, 0.5, ..., A(A-1) + 0.5 (CoETools.cpp:577-589) */
};
/* clustering.distance= : CoMap.cpp:401-427; Distance.h:150-173,316-424 */
enum { CMB_DIST_CORRELATION = 0, CMB_DIST_COMPENSATION = 1, CMB_DIST_EUCLIDIAN = 2 };
/* clustering.method= : CoMap.cpp:460-481 */
enum { CMB_LINK_COMPLETE = 0, CMB_LINK_SINGLE = 1, CMB_LINK_AVERAGE = 2 };

/* statistic.min_rate_class / .min_rate / .max_rate_class_diff / .max_rate_diff / .min,
 * CoETools.cpp:420-481; defaults 0, 0, -1, -1, 0 disable every filter. */
typedef struct cmb_filters {
  int32_t min_rate_class;
  int32_t max_rate_class_diff;
  double min_rate;
  double max_rate_diff;
  double min_stat;
} cmb_filters;

const char* cmb_last_error(void);
int cmb_version(void);

/* Pinned host memory for fast host<->device copies (optional convenience). */
int cmb_host_alloc(uint64_t bytes, void** out);
int cmb_host_free(void* p);

/* device < 0 uses the current device.  stream == NULL creates a private stream;
 * otherwise the given cudaStream_t (e.g. torch's current stream) is used. */
int cmb_ctx_create(int device, void* stream, cmb_ctx** out);
int cmb_ctx_destroy(cmb_ctx* ctx);
int cmb_sync(cmb_ctx* ctx);

/* Replaces the TreeTemplate<Node> handed to DRHomogeneousTreeLikelihood,
 * CoMap.cpp:125-126, CoETools.cpp:124. */
int cmb_set_tree(cmb_ctx* ctx, int32_t n_nodes, const int32_t* parent, const double* brlen);

/* Replaces model / rDist / substitutionCount (CoMap.cpp:136-152; CoETools.cpp:113,122).
 * Builds P_c(b) = exp(Q d_b r_c) and the count tables n_c(b) for every branch x class.
 * weight_xy: nullable A*A weights (AlphabetIndex2) of the weighted Total register. */
int cmb_set_model(cmb_ctx* ctx, int32_t A, const double* Q, const double* pi, int32_t C,
                  const double* rates, const double* probs, int32_t count_method,
                  const double* weight_xy);

/* Replaces tl->setData(*sites); tl->initialize() (CoETools.cpp:358-359). */
int cmb_set_alignment(cmb_ctx* ctx, int64_t S, const uint8_t* codes, int32_t n_codes,
                      const uint32_t* code_mask);

/* Replaces CoETools::getVectors -> LegacySubstitutionMappingTools::computeSubstitutionVectors
 * (CoETools.cpp:395-397), the norms loop (CoMap.cpp:158-163) and the per-site columns of
 * writeInfos (CoETools.cpp:507-510).  n_out is site-major [S][B] (mapping[i] is site i's
 * branch vector, Statistics.h:154-160); all outputs nullable.  The vectors stay resident
 * on the device for cmb_pairs / cmb_distance_matrix.
 * With EVERY output NULL the mapping is only enqueued (on a side stream, so that work enqueued next -- the
 * null replicates -- overlaps it: a 5000-site mapping is one latency-bound tree walk on a few SMs); the first
 * call that needs it waits for it and reports a saturated alignment (likelihood 0 at some site,
 * CoETools.cpp:233-262) then.  With any output requested the call completes the mapping and fails on
 * saturated sites after filling the per-site outputs. */
int cmb_map(cmb_ctx* ctx, double* n_out, double* norm, double* post_rate, int32_t* rate_class,
            double* loglik);

/* nijt.average / nijt.joint (CoETools.cpp:393-407 for the observed mapping, AnalysisTools.cpp:597-633 and
 * CoETools.cpp:1067-1082 for the simulated ones): which LegacySubstitutionMappingTools function fills the vectors
 * of every later mapping -- cmb_map, the null distributions, the candidates sampler; the clustering null always
 * averages (ClusterTools.cpp:227).  (1, 1) computeSubstitutionVectors (default, tensor-core kernels);
 * (1, 0) ...Marginal; (0, 1) ...NoAveraging; (0, 0) ...NoAveragingMarginal (thread-per-site kernels,
 * k1_variants.cu).  Invalidates the current mapping and null. */
int cmb_set_map_mode(cmb_ctx* ctx, int32_t average, int32_t joint);

/* asr.method = marginal (CoMap.cpp:168-198, a side output "not used in the analysis"): the state of largest marginal
 * posterior probability at every node of the tree for every site of the alignment -- LegacyMarginalAncestralState
 * Reconstruction::getAllAncestralStates [Bio++ / from memory: first arg-max over the states of sum_c p_c L_c(x) / L;
 * a leaf gets its first compatible state].  states is [n_nodes][S], node ids as in cmb_set_tree. */
int cmb_ancestral_states(cmb_ctx* ctx, uint8_t* states);

/* Restart path, input.vectors.file (CoETools.cpp:374-385): replaces the mapping computed by
 * cmb_map with vectors read from a file (site-major [S][B], as LegacySubstitutionMappingTools::
 * readFromStream yields them); site likelihoods, rates and rate classes stay those of the
 * alignment, as upstream.  norm (nullable) receives the norms of the loaded vectors. */
int cmb_load_vectors(cmb_ctx* ctx, const double* n_in, double* norm);

/* Replaces seqSim.simulate(n) (AnalysisTools.cpp:591,614; ClusterTools.cpp:224) in
 * discrete-rate mode with a counter-based Philox4x32-10 stream keyed
 * (seed, global site index, node).  weighted_classes = 0 draws the rate class uniformly
 * (upstream behaviour), 1 draws it from probs.  states is [T][n]; classes nullable. */
int cmb_simulate(cmb_ctx* ctx, uint64_t seed, int64_t first_site, int64_t n,
                 int32_t weighted_classes, uint8_t* states, int32_t* classes);

/* simulations.continuous = yes (CoMap.cpp:146,209-219: NonHomogeneousSequenceSimulator::enableContinuousRates):
 * every later simulation (cmb_simulate, the null distributions, the clustering null, the candidates sampler)
 * draws one rate per site from the continuous distribution -- kind 1 Constant, 2 Gamma(alpha, beta = alpha),
 * 3 Invariant(p) + Gamma(alpha) / (1 - p) -- and evolves the site with P(d_b r) computed on the fly, instead of
 * picking one of the discrete classes; classes are then reported as -1.  kind 0 restores the discrete classes.
 * The mapping of the simulated sites uses the discrete model either way, as upstream. */
int cmb_set_continuous_rates(cmb_ctx* ctx, int32_t kind, double alpha, double p_invariant);

/* Replaces AnalysisTools::getNullDistributionIntraDR (AnalysisTools.cpp:564-658) + the
 * per-bin sort (CoETools.cpp:650-652): rep_cpu x { simulate 2 x rep_ram sites, map both,
 * paired statistic j<->j, bin by Nmin in Domain(0, nmax, K) }.  Outer replicates
 * [rep_begin, rep_end) are computed (shard of a multi-GPU run; pass 0, rep_cpu for all);
 * site indices are global so results do not depend on the sharding.  raw (nullable) is
 * [(rep_end-rep_begin)*rep_ram][4] = Stat, RCmin, PRmin, Nmin
 * (statistic.null.output.file, AnalysisTools.cpp:642).  The binned, sorted null stays in
 * the context for cmb_pairs.  nmax < 0 uses max(norm) of the mapped alignment
 * (CoETools.cpp:640). */
int cmb_null_intra(cmb_ctx* ctx, int32_t stat_id, uint64_t seed, int32_t rep_cpu, int32_t rep_ram,
                   int32_t rep_begin, int32_t rep_end, int32_t weighted_classes, int32_t K,
                   double nmax, double* raw);

/* Multi-GPU (SURVEY.md s8e): one cmb_ctx per GPU, joined by an NCCL communicator that the library drives on
 * the context's stream (libnccl.so.2 is bound at run time; single-GPU use needs no NCCL).
 *   cmb_comm_unique_id / cmb_comm_init : one process per GPU -- rank 0 obtains the 128-byte id, the launcher
 *                        broadcasts it (MPI, torch.distributed, a file ...), every rank joins
 *   cmb_comm_init_all  : one process, n contexts on n distinct devices (the comap_b200 command line with
 *                        comap_b200.gpus=n); collective calls must then be issued from one thread per context
 *                        or between cmb_comm_group_start / _end
 *   cmb_comm_set       : adopt an ncclComm_t the caller already owns
 * The reference has no counterpart: it is single-threaded (CMakeLists.txt:5-19). */
int cmb_comm_unique_id(void* id128);
int cmb_comm_init(cmb_ctx* ctx, int32_t n_ranks, int32_t rank, const void* id128);
int cmb_comm_init_all(cmb_ctx** ctxs, int32_t n);
int cmb_comm_set(cmb_ctx* ctx, void* nccl_comm, int32_t n_ranks, int32_t rank);
int cmb_comm_destroy(cmb_ctx* ctx);
int cmb_comm_rank(cmb_ctx* ctx, int32_t* rank, int32_t* n_ranks);
int cmb_comm_group_start(void);
int cmb_comm_group_end(void);

/* cmb_null_intra over the communicator (AnalysisTools.cpp:564-658 sharded by outer replicate): this rank
 * simulates, maps and scores its contiguous share of the rep_cpu replicates (global site indices: the samples
 * do not depend on the rank count), the (Stat, Nmin) samples are all-gathered with ncclAllGather on the
 * context's stream, and every rank bins and sorts the union, so cmb_pairs on any shard of rows sees the same
 * null distribution as a single-GPU run.  Without a communicator it is cmb_null_intra over all replicates.
 * raw (nullable): the rows of THIS rank's replicates, [(r1 - r0) * rep_ram][4] with r0 = rank * q + min(rank, m),
 * r1 = r0 + q + (rank < m), q = rep_cpu / n_ranks, m = rep_cpu % n_ranks. */
int cmb_null_intra_sharded(cmb_ctx* ctx, int32_t stat_id, uint64_t seed, int32_t rep_cpu, int32_t rep_ram,
                           int32_t weighted_classes, int32_t K, double nmax, double* raw);

/* Parity hook: same as cmb_null_intra with the RNG bypassed.  sim1/sim2 are
 * [rep_cpu][T][rep_ram] state codes under the identity code table. */
int cmb_null_intra_from_alignments(cmb_ctx* ctx, int32_t stat_id, int32_t rep_cpu, int32_t rep_ram,
                                   const uint8_t* sim1, const uint8_t* sim2, int32_t K,
                                   double nmax, double* raw);

/* Threshold of CMB_STAT_MI (statistic=MI(threshold=0.99), CoETools.cpp:591): a branch entry is in
 * category 1 when it reaches the threshold. */
int cmb_set_mi_threshold(cmb_ctx* ctx, double threshold);

/* on = 1: cmb_null_intra with K = 0 (samples left unbinned for an exchange) only enqueues its
 * work and returns; the caller orders later consumers with cmb_sync.  Lets a second context on
 * another stream map and score the observed alignment while the null replicates run. */
int cmb_set_async(cmb_ctx* ctx, int32_t on);

/* Multi-GPU exchange step: the unbinned null samples of this context's shard live in
 * device memory; export them, all-gather with NCCL, then load the union into every rank. */
int cmb_null_samples_dev(cmb_ctx* ctx, const double** stat_dev, const double** nmin_dev,
                         int64_t* n);
int cmb_null_load_dev(cmb_ctx* ctx, const double* stat_dev, const double* nmin_dev, int64_t n,
                      int32_t K, double nmax);
/* Sorted per-bin null: bin_offsets [K+1], sorted [bin_offsets[K]] (both nullable). */
int cmb_null_get(cmb_ctx* ctx, int32_t* K, double* nmax, int64_t* bin_offsets, double* sorted,
                 int64_t capacity);

/* Replaces the pair loop of CoETools::computeIntraStats (CoETools.cpp:672-724): all pairs
 * i<j of the mapped alignment, filters, p = (nsim - #{sim < stat} + 1)/(nsim + 1) in the
 * Nmin bin, NaN / 0 when Nmin is outside [0, nmax) (the "NA\t0" rows).  Rows come out in
 * the reference's order (i ascending, then j).  Only rows i with
 * i % (2*shard_count) in {shard_index, 2*shard_count-1-shard_index} are produced
 * (shard_count = 1: all rows).  use_null = 0 skips the p-value columns.  Every output
 * column is nullable; capacity is in rows. */
int cmb_pairs(cmb_ctx* ctx, int32_t stat_id, const cmb_filters* filters, int32_t use_null,
              int32_t shard_index, int32_t shard_count, int64_t capacity, int32_t* out_i,
              int32_t* out_j, double* out_stat, int32_t* out_rcmin, double* out_prmin,
              double* out_nmin, double* out_pvalue, int32_t* out_nsim, int64_t* n_rows);

/* Device-resident form of cmb_pairs: computes the columns selected by the bitmask
 * `columns` (bit k = column k: 0 i, 1 j, 2 stat, 3 rcmin, 4 prmin, 5 nmin, 6 pvalue,
 * 7 nsim, int32) into device memory and returns the row count; cmb_pairs_fetch then copies one
 * column to the host (asynchronously on the context's stream; call cmb_sync). */
int cmb_pairs_resident(cmb_ctx* ctx, int32_t stat_id, const cmb_filters* filters, int32_t use_null,
                       int32_t shard_index, int32_t shard_count, uint32_t columns, int64_t* n_rows);
int cmb_pairs_fetch(cmb_ctx* ctx, int32_t column, void* host, int64_t capacity);

/* Two data sets on the same tree topology ("inter-gene" analysis), one context each.
 * Replaces CoETools::computeInterStats (CoETools.cpp:732-840): the statistic of every site i of
 * data set 1 with every site j of data set 2 -- or of site i with site i when `independent`
 * (independant_comparisons, CoETools.cpp:744-749,795-796) -- in the reference's row order (i, then
 * j).  `filters` holds data set 1's rate thresholds and the shared ones; min_rate_class2 /
 * min_rate2 are statistic.min_rate_class2 / .min_rate2 (CoETools.cpp:757-761).  nmin_by_row = 1
 * reproduces upstream's Nmin = min(norms1[i], norms2[i]) (CoETools.cpp:803), 0 pairs norms2[j].
 * No p-values upstream for this analysis.  Every output column is nullable. */
int cmb_pairs_inter(cmb_ctx* ctx1, cmb_ctx* ctx2, int32_t stat_id, const cmb_filters* filters,
                    int32_t min_rate_class2, double min_rate2, int32_t independent, int32_t nmin_by_row,
                    int64_t capacity, int32_t* out_i, int32_t* out_j, double* out_stat, int32_t* out_rcmin,
                    double* out_prmin, double* out_nmin, int64_t* n_rows);

/* Replaces AnalysisTools::getNullDistributionInterDR (AnalysisTools.cpp:662-735;
 * CoETools.cpp:878-897): rep_cpu x { simulate rep_ram sites under each data set's own tree /
 * model / rate distribution, map both, paired statistic j<->j }.  raw is
 * [rep_cpu*rep_ram][4] = Stat, RCmin, PRmin, Nmin (statistic.null.output.file).  Data set 2
 * draws from the stream keyed seed ^ 0x9E3779B97F4A7C15 at the same site indices. */
int cmb_null_inter(cmb_ctx* ctx1, cmb_ctx* ctx2, int32_t stat_id, uint64_t seed, int32_t rep_cpu,
                   int32_t rep_ram, int32_t weighted_classes, double* raw);
/* cmb_null_inter over the outer replicates [rep_begin, rep_end) only (one GPU's share of a multi-GPU
 * run; cmb_null_inter is the range [0, rep_cpu)).  raw is [(rep_end-rep_begin)*rep_ram][4], the rows of
 * the whole call for those replicates bit for bit: both simulators are keyed by the global site index. */
int cmb_null_inter_range(cmb_ctx* ctx1, cmb_ctx* ctx2, int32_t stat_id, uint64_t seed, int32_t rep_cpu,
                         int32_t rep_ram, int32_t rep_begin, int32_t rep_end, int32_t weighted_classes,
                         double* raw);

/* Candidate groups (analysis=candidates): replaces CandidateGroup::computeStatisticValue /
 * computeNormRanges (CoMap.cpp:663-667; CoETools.h:106-128) and
 * CoETools::computePValuesForCandidateGroups + CandidateGroupSet::analyseSimulations
 * (CoETools.cpp:901-1087).  Group g = sites group_sites[group_off[g] .. group_off[g+1]) of the
 * mapped alignment; analysable (nullable) marks groups to test.  Batches of rep_ram sites are
 * simulated and mapped until every analysable group has min_sim simulated groups (sites dealt to
 * candidate sites whose norm lies within +-omega, upstream's iteration order) or max_trials
 * batches completed no group.  out_stat: observed group statistic (minimum over pairs, or the
 * compensation group formula); out_pvalue = (n1 + 1) / (n2 + 1); all outputs nullable. */
int cmb_candidates(cmb_ctx* ctx, int32_t stat_id, int32_t n_groups, const int64_t* group_off,
                   const int32_t* group_sites, const uint8_t* analysable, double omega, int64_t min_sim,
                   int32_t max_trials, int32_t rep_ram, uint64_t seed, int32_t weighted_classes,
                   double* out_stat, double* out_pvalue, int64_t* out_n1, int64_t* out_n2,
                   int64_t* n_simulated);

/* Replaces the distance-matrix loop (CoMap.cpp:432-440; ClusterTools.cpp:242-251).
 * mat (nullable) receives the full symmetric S*S matrix; it also stays on the device. */
int cmb_distance_matrix(cmb_ctx* ctx, int32_t dist_id, double* mat);

/* Replaces HierarchicalClustering(method, mat, false) + computeTree (CoMap.cpp:460-485;
 * ClusterTools.cpp:260-262) on the resident distance matrix (consumed).  Dendrogram:
 * leaves 0..S-1, inner nodes S..2S-2 in creation order; left/right/height [S-1],
 * height = merge distance / 2. */
int cmb_cluster(cmb_ctx* ctx, int32_t linkage, int32_t* left, int32_t* right, double* height);

/* Replaces ClusterTools::getGroups + computeNormProperties + Distance::setStatisticAsProperty
 * and the size filter (CoMap.cpp:488-545; ClusterTools.cpp:59-113,296-319;
 * Distance.h:109-129,346-368,390-422) on the last dendrogram.  members: flat, capacity
 * (S-1)*max_size; offsets [S]; g_* [S-1]. */
int cmb_groups(cmb_ctx* ctx, int32_t dist_id, int32_t max_size, int32_t* members, int64_t* offsets,
               double* g_height, double* g_stat, double* g_nmin, int64_t* n_groups);

/* Replaces ClusterTools::computeGlobalDistanceDistribution (ClusterTools.cpp:200-294):
 * replicates [rep_begin, rep_end) of { simulate S sites, map, distance matrix, cluster,
 * groups <= max_size }.  Rows: rep, size, Dmax = 2*height, Stat, Nmin, and the member
 * matrix indices (flat + offsets).  capacity_rows / capacity_members bound the outputs.
 * Up to four replicates are clustered by one launch (each holds its own S x S matrix on the
 * device while it does; fewer when memory is short); results do not depend on the batching. */
int cmb_cluster_null(cmb_ctx* ctx, int32_t dist_id, int32_t linkage, uint64_t seed,
                     int32_t rep_begin, int32_t rep_end, int32_t weighted_classes, int32_t max_size,
                     int64_t capacity_rows, int64_t capacity_members, int32_t* row_rep,
                     int32_t* row_size, double* row_dmax, double* row_stat, double* row_nmin,
                     int32_t* members, int64_t* offsets, int64_t* n_rows);

/* ---- Mica (CoMap/Mica.cpp): mutual information between alignment COLUMNS, conditioned like the pairwise analysis ----
 * SiteTools::entropy / mutualInformation / jointEntropy(site, resolveUnknowns = true) are Bio++ bpp-seq code that is not
 * in the reference tree and no output of mica ships with it: restated from memory, parity unpinned. */
enum { CMB_MICA_KEY_NMIN = 1 /* use_model = yes: bins of min(norm), Mica.cpp:397 */, CMB_MICA_KEY_HMIN = 2 /* bins of min(entropy), :399 */ };
/* Mica.cpp:341-361: entropy of every site and its average MI with all the other sites (nullable outputs, [S]). */
int cmb_mica_sites(cmb_ctx* ctx, double* entropy, double* average_mi);
/* The table loop, Mica.cpp:646-689: all pairs i < j in that order -- MI, joint entropy, Hmin = min(entropy), Nmin = min
 * norm of the mapped alignment (NaN without cmb_map) and, with use_null, the p-value (nsim - #{sim < MI} + 1)/(nsim + 1)
 * in the bin of `key` (NaN / 0 where mica prints "NA 0").  APC and RCW are averageMI[i] averageMI[j] / mean(averageMI)
 * and / 2 (:661-662): one multiplication per row, left to the caller. */
int cmb_mica_pairs(cmb_ctx* ctx, int32_t key, int32_t use_null, int64_t capacity, int32_t* out_i, int32_t* out_j, double* mi,
                   double* hjoint, double* hmin, double* nmin, double* pvalue, int32_t* nsim, int64_t* n_rows);
/* MI / joint entropy of listed site pairs of the alignment: the nonparametric bootstrap's resampled pairs (Mica.cpp:423-431). */
int cmb_mica_pair_list(cmb_ctx* ctx, int64_t n, const int32_t* site1, const int32_t* site2, double* mi, double* hjoint);
/* null.method = permutations (miTest, Mica.cpp:92-118; table columns Perm.p.value / Perm.nb, :666-667): for every pair, in
 * the order of cmb_mica_pairs, both columns are shuffled until 5 shuffled MIs reach the observed one or max_permutations
 * were drawn; pvalue = (count + 1) / (shuffles + 1), nperm = shuffles; 1 and 0 when a column is constant.  Upstream's
 * generator is unseeded and its copies are reshuffled in place; here every shuffle is drawn from the original columns
 * (the same distribution) and is a function of (seed, pair, shuffle number) only -- see DESIGN.md s4 K5. */
int cmb_mica_permutations(cmb_ctx* ctx, uint64_t seed, int32_t max_permutations, int64_t capacity, double* pvalue, int32_t* nperm,
                          int64_t* n_rows);
/* One shard of cmb_mica_permutations (one GPU's share of a multi-GPU run; needs no communicator): the pairs
 * idx = shard_index + k shard_count, k = 0, 1, ... of cmb_mica_pairs' order, row k of the outputs holding pair idx.  Each
 * row is bit for bit the row idx of cmb_mica_permutations (shard_count = 1).  0 <= shard_index < shard_count; a shard
 * past the last pair has 0 rows.  The shards interleave so that each gets its part of the pairs that run all their
 * shuffles, wherever they sit in the table. */
int cmb_mica_permutations_shard(cmb_ctx* ctx, uint64_t seed, int32_t max_permutations, int32_t shard_index, int32_t shard_count,
                                int64_t capacity, double* pvalue, int32_t* nperm, int64_t* n_rows);
/* null.method = parametric-bootstrap (Mica.cpp:470-545): per outer replicate two simulated alignments of rep_ram sites,
 * mapped for their norms (computeSubstitutionVectors), MI of site j with site j, binned by min norm over [0, nmax)
 * (nmax < 0: the mapped alignment's largest norm).  raw: nullable [rep_cpu * rep_ram][3] = MI, Hjoint, Nmin. */
int cmb_mica_null_parametric(cmb_ctx* ctx, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t weighted_classes, int32_t K,
                             double nmax, double* raw);
/* cmb_mica_null_parametric over the outer replicates [rep_begin, rep_end) (cmb_mica_null_parametric is [0, rep_cpu)):
 * raw holds this range's [(rep_end - rep_begin) * rep_ram][3] rows, and K > 0 bins this range's samples only.  Replicate r
 * simulates the global sites from 2 r rep_ram, so the ranges concatenate to the whole null. */
int cmb_mica_null_parametric_range(cmb_ctx* ctx, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t rep_begin,
                                   int32_t rep_end, int32_t weighted_classes, int32_t K, double nmax, double* raw);
/* cmb_mica_null_parametric over the communicator, as cmb_null_intra_sharded: this rank scores its contiguous share of the
 * replicates (the r0, r1 documented there), the (MI, Nmin) samples are all-gathered, and every rank bins and sorts the
 * union, so cmb_mica_pairs on any rank sees the single-GPU null.  raw (nullable): the rows of THIS rank's replicates.
 * K = 0: no binning and no exchange.  Without a communicator it is cmb_mica_null_parametric. */
int cmb_mica_null_parametric_sharded(cmb_ctx* ctx, uint64_t seed, int32_t rep_cpu, int32_t rep_ram, int32_t weighted_classes,
                                     int32_t K, double nmax, double* raw);
/* A null distribution from host arrays -- n statistics and the key they are conditioned on, K bins over [0, kmax) -- for
 * the null methods whose samples the caller builds (Mica.cpp:401-468 nonparametric bootstrap, :546-606 z-score). */
int cmb_null_load(cmb_ctx* ctx, const double* stat, const double* key, int64_t n, int32_t K, double kmax);

/* Measurement: device time (CUDA events on the context's stream) and launch counts per
 * kernel family since the last reset.  name in {"map_down","map_up","simulate","pairs",
 * "null_pairs","sort","distance","cluster","other"}. */
int cmb_profile_enable(cmb_ctx* ctx, int32_t on);
int cmb_profile_reset(cmb_ctx* ctx);
int cmb_profile_get(cmb_ctx* ctx, const char* name, double* ms, int64_t* launches);
int64_t cmb_launch_count(cmb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
