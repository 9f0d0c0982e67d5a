/* tlc_b200.h -- C-ABI of libtlc_b200.so: the B200 (sm_100a) implementation of TLC-GNN's per-target
 * topological feature path (vicinity -> filtration -> 0-dim ordinary/extended persistence [+ 1-dim
 * loops] -> persistence image).
 *
 * The reference (pkuyzy/TLC-GNN) has no FFI: its boundary is the Python package `sg2dgm`.  Each entry
 * point below names the reference interface it replaces (paths relative to the reference root); the
 * Python mirror in tlc-gnn_b200/sg2dgm/ binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only.  "host" pointers are ordinary host memory, "dev"
 * pointers are CUDA device memory on the graph's device.  Every function returns 0 on success or a
 * negative tlc_rc; tlc_last_error() returns a thread-local message for the last failure.
 * Per-target outcomes never fail a call: they are reported in a uint8 status array
 * (riccidist2dgm.py:352-357 swallows per-edge exceptions into zero rows).
 */
#ifndef TLC_B200_H
#define TLC_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes ---- */
#define TLC_OK 0
#define TLC_E_INVALID (-1) /* bad argument */
#define TLC_E_CUDA (-2)    /* CUDA runtime error (message has the cudaError string) */
#define TLC_E_NOMEM (-3)   /* host or device allocation failed / one vicinity exceeds the arena */
#define TLC_E_NODEVICE (-4)
#define TLC_E_CAPACITY (-5) /* caller-provided output capacity too small */

/* ---- vicinity mode ---- */
#define TLC_MODE_EDGE 0 /* ball(u) & ball(v), induced          riccidist2dgm.py:311-316 */
#define TLC_MODE_NODE 1 /* ball(u) (PDGNN generators)          Knowledge_Distillation/data_utils_NC.py:97-100 */
#define TLC_MODE_EDGE_FORCED 2 /* (ball(u) & ball(v)) + {u, v}: the PDGNN link-prediction generator's vicinity, the two
                                  roots always members; no edge at all -> TLC_ST_EMPTY (`return None, None`)
                                  Knowledge_Distillation/data_utils_LP.py:107-118 */

#define TLC_MODE_EDGE_UNION 3 /* ball(u) | ball(v): `range == 'union'` of the legacy sg2pimg   riccidist2dgm.py:242-247 */
#define TLC_MODE_EDGE_REMOVEINTER 4 /* (ball(u) | ball(v)) - (ball(u) & ball(v)) + [u, v]: `range == 'removeinter'`   :289-296 */

/* ---- descriptor: which node attribute is the filtration     riccidist2dgm.py:47-49 ---- */
#define TLC_DESC_MIN 0
#define TLC_DESC_MAX 1
#define TLC_DESC_SUM 2

/* ---- flags ---- */
#define TLC_F_NORM 1u       /* build_fv(norm=True)                       riccidist2dgm.py:50-56 */
#define TLC_F_EXTENDED 2u   /* + Accelerate_PD (1-dim extended pairs)    riccidist2dgm.py:323-326 */
#define TLC_F_KEEP_ZERO 4u  /* KD copy: emit zero-persistence pairs      KD/accelerated_PD.py:68-69,108-109,169-170 */
#define TLC_F_NORM_EPS 8u   /* KD: divide by (max + 1e-10)               KD/data_utils_NC.py:54 */
#define TLC_F_SUM_PLAIN 16u /* path sums left-to-right (CPython <= 3.11); default Neumaier (CPython >= 3.12 sum()) */
#define TLC_F_EDGE_SORTED 32u /* ascending sweep by the edge-sorted kernels 2+3 for every target (default: the
                                 vertex-ordered kernels 2v+3v, which produce the identical pair sequence and hand
                                 targets they cannot finish to kernels 2+3) -- a test/diagnostic switch */

#define TLC_F_NO_DIRECT 64u /* never take the graph-row route (below): always materialise the induced adjacency */
#define TLC_F_DIRECT 128u   /* take the graph-row route whatever the density.  Default: per call, when its vicinities
                               are dense in the graph (sum of their graph degrees <= TLC_DIRECT_RATIO (env, default 2)
                               x their induced directed edges): the filtration, vertex order and sweep kernels then
                               read the graph's own L2-resident CSR rows through the vicinity bitmap instead of an
                               adjacency written to HBM.  Same results bit for bit; only taken by calls that need
                               the ascending sweep alone (no TLC_F_EXTENDED, no Pos/Neg lists) */
#define TLC_F_ASC_ONLY 256u /* tlc_vicinity_detail: ascending sweep only -- PD_up and [min,max]; no PD_down, no edge
                               lists / orders / Pos / Neg (those outputs are left untouched) */

#define TLC_F_NO_SMALL 4096u /* never take the fused small-vicinity kernels (kernel S): every target through the staged
                                pipeline.  Default: the batch calls (5 x 5 image, Ricci-distance filtration) first run kernel S,
                                which finishes every vicinity of <= 1024 vertices / <= 4096 edges in one launch per size class,
                                and hand only the larger ones to the staged kernels.  Same results bit for bit */

#define TLC_F_NO_TABLE 8192u /* graph-row route: never use the per-root shortest-path tables (kernel 1t), always run kernel 1b's
                                Dijkstra per target.  Default: on graphs of <= 16384 nodes whose tables fit the budget
                                (28 N^2 bytes <= TLC_SSSP_CACHE_GB GiB, default 8) the distances, tree parents and path sums of
                                a root over its k-hop ball are computed once; a vicinity vertex whose tree branch stays inside
                                the vicinity takes its values from the table, the others are relaxed over their own rows.
                                Same results bit for bit */

#define TLC_F_FILT_DEGREE 512u      /* PDGNN generators, filt='degree': filtration = induced degree / (max + 1e-10)
                                       Knowledge_Distillation/data_utils_NC.py:126-128 (no roots, no distances) */
#define TLC_F_FILT_CENTRALITY 1024u /* filt='centrality': nx.degree_centrality (d * 1/(n-1)) / (max + 1e-10)   :118-121 */
#define TLC_F_FILT_CLUSTERING 2048u /* filt='clustering': nx.clustering (2 T / (d (d-1))) / (max + 1e-10)      :122-125 */

#define TLC_F_FILT_HKS 16384u /* filt='hks' (the PDGNN generators' default): heat kernel signature of the UNWEIGHTED vicinity,
                                  hks(x) = sum_k exp(-t lambda_k) phi_k(x)^2 = [exp(-t L)]_xx, L the symmetric normalised
                                  Laplacian, divided by (max + 1e-10)   Knowledge_Distillation/data_utils_NC.py:87-93,115-117.
                                  t = tlc_graph_set_hks_time (default 0.1).  The reference diagonalises L (scipy eigh); the
                                  kernel evaluates the same diagonal through the Taylor series of exp((t/2) N) e_x, N = I - L:
                                  float64, agreement ~1e-13 -- values are not bit-identical to a LAPACK run (nor is LAPACK to
                                  itself across builds), so this filtration is pinned to 1e-9, not bit for bit */
#define TLC_F_FILT_ANY_STRUCT (TLC_F_FILT_DEGREE | TLC_F_FILT_CENTRALITY | TLC_F_FILT_CLUSTERING | TLC_F_FILT_HKS)

/* ---- pair kinds, in the reference's concatenation order    accelerated_PD.py:110, riccidist2dgm.py:328 ---- */
#define TLC_K_UP 0      /* PD_up   : 0-dim ordinary                 accelerated_PD.py:65-66 */
#define TLC_K_ESS 1     /* [min,max]                                accelerated_PD.py:110   */
#define TLC_K_DOWN 2    /* PD_down : relative                       accelerated_PD.py:105-106 */
#define TLC_K_ESS_REV 3 /* [max,min]                                accelerated_PD.py:110   */
#define TLC_K_ONE 4     /* PD_one  : 1-dim extended (loops)         accelerated_PD.py:164-165 */

/* ---- per-target status (SURVEY.md A.8) ---- */
#define TLC_ST_OK 0
#define TLC_ST_TRIVIAL 1        /* roots outside the vicinity: all values equal, image zero, counted */
#define TLC_ST_EMPTY 2          /* empty vicinity                          riccidist2dgm.py:318 */
#define TLC_ST_DISCONNECTED 3   /* >1 component                            riccidist2dgm.py:318 */
#define TLC_ST_DEGENERATE 4     /* normaliser 0 (vicinity == {u,v})        riccidist2dgm.py:54-56 */
#define TLC_ST_UNKNOWN_NODE 5   /* id not in the graph / isolated          riccidist2dgm.py:353 */
#define TLC_ST_BAD_DESCRIPTOR 6 /* attribute missing                       accelerated_PD.py:13 */
#define TLC_ST_NO_TREE_EDGES 7  /* single vertex + extended flag           accelerated_PD.py:122 */
#define TLC_ST_NONFINITE 8      /* tlc_graph_batch_diagrams_dev: a NaN or +-inf filtration value, no pairs */

typedef struct {
  int32_t hop;        /* BFS depth limit                                   riccidist2dgm.py:310 */
  int32_t mode;       /* TLC_MODE_*                                                             */
  int32_t descriptor; /* TLC_DESC_*                                                             */
  int32_t resolution; /* image is resolution x resolution (1..16)          PersistenceImager.pyx:207 */
  uint32_t flags;     /* TLC_F_*                                                                */
  uint32_t img_mask;  /* bit k set: pairs of kind k are rasterised                              */
} tlc_params;

typedef struct tlc_graph tlc_graph; /* opaque: CSR + curvature resident in HBM, scratch arena, stream */

/* graph2pi.__init__ (riccidist2dgm.py:216-226): node ids are the reference's integer relabelling
 * (first appearance order); rowptr[N+1], col[nnz] ascending inside each row, kappa[nnz] = Ricci
 * curvature of the directed edge (weight = kappa + 1, :225).  All host pointers; copied to `device`.
 * The CSR is validated (TLC_E_INVALID otherwise): rowptr monotone, col in [0, N), rows strictly ascending (no
 * duplicate entries), no self-loops, every entry (x, y) mirrored by (y, x) with the same kappa, and kappa + 1 finite
 * and > 0 (the precondition of the reference's Dijkstra, SURVEY.md F1/F5).
 * arena_bytes = 0 picks a default (TLC_ARENA_GB env or 24 GiB, clamped to free memory). */
int tlc_graph_create(int32_t N, int64_t nnz, const int32_t *rowptr, const int32_t *col, const double *kappa,
                     int device, uint64_t arena_bytes, tlc_graph **out);
int tlc_graph_destroy(tlc_graph *g);

/* graph2pi.get_pimg_for_all_edges (riccidist2dgm.py:362-370) for a whole batch, HOST buffers.
 * targets[E][2] are graph ids (-1 = label unknown to dict_node).  out_pi[E][res*res] float64 rows
 * (zero for failed targets, as :363 pre-zeroes), out_status[E] (may be NULL), *cnt_compute (may be
 * NULL) = number of targets the reference would have counted (:354). */
int tlc_vicinity_pi(tlc_graph *g, const int32_t *targets, int64_t E, const tlc_params *p, double *out_pi,
                    uint8_t *out_status, int64_t *cnt_compute);

/* same, DEVICE buffers (inputs already resident; no host<->device copies of payload).
 * dev_out_pi is float64[E][res*res]; dev_out_pi_f32 (may be NULL) additionally receives float32
 * rows (the layout that is all-gathered across GPUs). */
int tlc_vicinity_pi_dev(tlc_graph *g, const int32_t *dev_targets, int64_t E, const tlc_params *p, double *dev_out_pi,
                        float *dev_out_pi_f32, uint8_t *dev_out_status, int64_t *cnt_compute);

/* vicinity sizes only (kernel 1, counting pass): n[E] vertices, m[E] induced edges, host buffers.
 * Lets a caller size diagram buffers: pairs(e) <= n + m + 1. */
int tlc_vicinity_sizes(tlc_graph *g, const int32_t *targets, int64_t E, const tlc_params *p, int32_t *out_n,
                       int32_t *out_m, uint8_t *out_status);

/* every intermediate of the path for a (small) batch, HOST buffers, for stage-level parity:
 *   voff[E+1], eoff[E+1], poff[E+1]  : exclusive offsets of the per-target segments
 *   vert[sum n]   graph ids ascending                     (kernel 1; riccidist2dgm.py:311-316)
 *   elo,ehi[sum m] local ids, lexicographic; ew = kappa+1 (kernel 1)
 *   fval[sum n]   filtration values                       (kernel 1b; riccidist2dgm.py:20-61)
 *   ord_asc, ord_desc[sum m] edge index in sweep order    (kernel 2; accelerated_PD.py:40-41,76-77)
 *   pairs: npairs[E]; pkind/pbv/pdv/pbirth/pdeath at poff (kernel 3/3b; local vertex ids)
 *   pos/neg edge indices in sweep order at eoff / voff; npos[E], nneg[E]
 *   pi[E][res*res], status[E]; pi_up / pi_one[E][res*res]: images of the kind-0 / kind-4 pairs alone
 * Any output pointer may be NULL.  cap_v/cap_e/cap_p are the capacities of the segment buffers
 * (TLC_E_CAPACITY if exceeded; use tlc_vicinity_sizes first). */
typedef struct {
  int64_t cap_v, cap_e, cap_p;
  int64_t *voff, *eoff, *poff;
  int32_t *n, *m, *lu, *lv, *npairs, *npos, *nneg;
  int32_t *vert, *elo, *ehi;
  double *ew, *fval;
  int32_t *ord_asc, *ord_desc;
  int32_t *pkind, *pbv, *pdv;
  double *pbirth, *pdeath;
  int32_t *pos, *neg;
  double *pi;
  uint8_t *status;
  /* PDGNN generator images (Knowledge_Distillation/data_utils_NC.py:172-176): the image of the PD_up pairs alone
   * (PI0 = transform(dgmOrd0)) and of the 1-dim extended pairs alone (PI1 = transform(dgmExt1)), [E][res*res] */
  double *pi_up, *pi_one;
} tlc_detail;
int tlc_vicinity_detail(tlc_graph *g, const int32_t *targets, int64_t E, const tlc_params *p, tlc_detail *out);

#define TLC_ST_NOT_SMALL 255 /* tlc_small_diagrams only: the vicinity exceeds kernel S (> 1024 vertices or > 4096 edges) */

/* Diagrams of a batch straight from the fused small-vicinity kernels (kernel S, k0_small.cu): for every target whose
 * vicinity has <= 1024 vertices and <= 4096 edges, the reference's PD_zero (+ PD_one with TLC_F_EXTENDED) in its own
 * concatenation order (accelerated_PD.py:110, riccidist2dgm.py:323-328) -- kind, birth / death vertex (local ids),
 * birth / death value -- at poff[t] .. poff[t] + npairs[t], plus the image row, status and vicinity size.  poff[E+1]
 * are the caller's exclusive segment offsets; a segment must hold n + m + 2 pairs (tlc_vicinity_sizes).  Targets
 * kernel S cannot take report TLC_ST_NOT_SMALL and no pairs (tlc_vicinity_detail serves those).  HOST buffers;
 * any output pointer may be NULL.  5 x 5 image, Ricci-distance filtration only. */
int tlc_small_diagrams(tlc_graph *g, const int32_t *targets, int64_t E, const tlc_params *p, const int64_t *poff,
                       int32_t *npairs, int32_t *pkind, int32_t *pbv, int32_t *pdv, double *pbirth, double *pdeath,
                       double *out_pi, uint8_t *out_status, int32_t *out_n, int32_t *out_m);

/* Persistence diagrams of a whole batch, on every route the batch call takes (kernel S, the materialised and the
 * graph-row route, chunking, sub-calls): graph2pi.get_pimg_for_all_edges' diagrams before the imager.  Target t's diagram
 * is np.array(PD0 + PD1) of riccidist2dgm.py:323-328 in that order -- PD_up, [min,max], PD_down, [max,min], then PD_one
 * with TLC_F_EXTENDED -- at poff[t] .. poff[t+1], in TARGET order.  TLC_F_ASC_ONLY (not with TLC_F_EXTENDED) keeps PD_up and
 * [min,max], the pairs of nonzero image weight without extended persistence, and lets the call take the graph-row route.
 * Every other flag keeps its batch-call meaning.  bv / dv are GRAPH ids (tlc_graph_create numbering).  Targets whose
 * status is neither OK, TRIVIAL nor NO_TREE_EDGES have no pairs.
 * Capacity: poff, npairs, *total_pairs, the image rows and the statuses are always written; if *total_pairs > cap the
 * call returns TLC_E_CAPACITY and leaves the pair arrays untouched (cap = 0: a sizing call; again with cap = *total_pairs
 * it succeeds).  Output is bit-identical from run to run; image rows and statuses equal tlc_vicinity_pi_dev's. */
typedef struct {
  int64_t cap;            /* capacity of the pair arrays, in pairs                                   */
  int64_t *poff;          /* [E+1] exclusive offsets, target order (required)                        */
  int32_t *npairs;        /* [E]   pairs per target (may be NULL)                                    */
  uint8_t *kind;          /* [cap] TLC_K_*                                  any of these may be NULL */
  int32_t *bv, *dv;       /* [cap] birth / death vertex, graph ids                                   */
  double *birth, *death;  /* [cap]                                                                   */
} tlc_diagrams;
/* DEVICE buffers: targets, every array of *out, dev_out_pi float64[E][res*res] (may be NULL), dev_out_status (may be NULL) */
int tlc_vicinity_diagrams_dev(tlc_graph *g, const int32_t *dev_targets, int64_t E, const tlc_params *p, tlc_diagrams *out,
                              double *dev_out_pi, uint8_t *dev_out_status, int64_t *total_pairs);
/* same, HOST buffers */
int tlc_vicinity_diagrams(tlc_graph *g, const int32_t *targets, int64_t E, const tlc_params *p, tlc_diagrams *out,
                          double *out_pi, uint8_t *out_status, int64_t *total_pairs);

/* compute_ricci_curvature (loaddatas.py:105-123): OllivierRicci(G, alpha, method="Sinkhorn").compute_ricci_curvature() on the
 * unweighted graph given as a symmetric CSR (ascending rows, no self-loops) -- the step BEFORE the path, whose output is
 * the `kappa` of tlc_graph_create.  out_kappa[nnz] receives the curvature of every directed entry (both directions of an
 * edge carry the same value, :117-121); out_iters[nnz] (may be NULL) the Sinkhorn iterations spent.  HOST buffers; runs
 * kernel 6 (k6_ricci.cu) on `device`.  The reference's arithmetic for this step lives in GraphRicciCurvature + POT, neither
 * vendored nor pinned by the reference: their published algorithm is restated (nbr_topk = 3000, reg = 0.1, <= 1000
 * iterations, stop at 1e-9) -- parity unpinned, see oracle/ricci_oracle.py. */
int tlc_ollivier_ricci(int device, int32_t N, int64_t nnz, const int32_t *rowptr, const int32_t *col, double alpha,
                       double *out_kappa, int32_t *out_iters);

/* Union_find(simplex_filter) + Accelerate_PD(Pos, Neg, simplex_filter) on ONE caller-supplied graph
 * (accelerated_PD.py:26,115; KD/accelerated_PD.py:25,120): n vertices with filtration fval[n], m edges
 * (a[i], b[i]) in the caller's dict order (that order is the tie-break).  flags: TLC_F_EXTENDED,
 * TLC_F_KEEP_ZERO.  Outputs as in tlc_detail (pairs capacity n+m+1; pos capacity m; neg capacity n).
 * Host buffers; runs kernels 2, 3, 3b on `device`. */
int tlc_union_find(int device, int32_t n, int32_t m, const double *fval, const int32_t *a, const int32_t *b,
                   uint32_t flags, int32_t *npairs, int32_t *pkind, int32_t *pbv, int32_t *pdv, double *pbirth,
                   double *pdeath, int32_t *npos, int32_t *pos, int32_t *nneg, int32_t *neg, uint8_t *status);

/* PersistenceImager(resolution).transform(dgm, skew=True) (PersistenceImager.pyx:352-388): host
 * dgm[K][2] (birth, death) float64 -> out[res*res] float64, runs kernel 4 on `device`. */
int tlc_pimg_transform(int device, const double *dgm, int64_t K, int32_t resolution, double *out);

/* The same imager for a batch of D diagrams already on the device, and its gradient: the batched form of
 * Knowledge_Distillation/pimg.py `transform` (:354-414), the torch copy of PersistenceImager(resolution).transform(dgm,
 * skew=True) (PersistenceImager.pyx:352-388) that PDGNN differentiates through.  Diagram t is the points
 * poff[t] .. poff[t+1] of birth[] / death[]; poff[0] need not be 0 (a slice of a larger diagram array works).  poff must be
 * non-decreasing with every entry in [0, len(birth)]: a decreasing segment is treated as empty, and no point outside
 * [poff[t], poff[t+1]) is read for diagram t.  kind (may be NULL: every point counts) selects the points whose kind k is
 * < 32 with bit k of img_mask set.  out[D][res*res] float64, birth-major; an empty diagram gives a zero row.
 * Gradient: with p = death - birth, w = clamp(p, 0, 1), A_i(b) = Phi(x_{i+1} - b) - Phi(x_i - b), B_j(p) likewise and
 * G = grad_out[t]:  grad_death = A^T G (w' B + w B'),  grad_birth = w A'^T G B - grad_death,  where w' = 1 on the CLOSED
 * interval 0 <= p <= 1 and 0 elsewhere (torch.clamp's own backward), so zero-persistence points get a nonzero
 * grad_death.  Points whose kind is masked out get 0.  grad_birth[k] / grad_death[k] are written for every k in
 * [poff[0], poff[D]) and nowhere else; either pointer may be NULL (not computed).
 * Every pointer is a DEVICE pointer on `device`; `stream` is a cudaStream_t (NULL: default stream).  Neither call
 * allocates or synchronises: both only enqueue.  Results are bit-identical from call to call and independent of the
 * rest of the batch (a batch split over sliced poff gives the same rows).  TLC_E_INVALID: D outside [0, 2^31),
 * resolution outside 1..16, or a NULL required pointer with D > 0. */
int tlc_pimg_batch_dev(int device, int64_t D, const int64_t *dev_poff, const double *dev_birth, const double *dev_death,
                       const uint8_t *dev_kind, uint32_t img_mask, int32_t resolution, double *dev_out, void *stream);
int tlc_pimg_batch_grad_dev(int device, int64_t D, const int64_t *dev_poff, const double *dev_birth,
                            const double *dev_death, const uint8_t *dev_kind, uint32_t img_mask, int32_t resolution,
                            const double *dev_grad_out, double *dev_grad_birth, double *dev_grad_death, void *stream);

/* Exact Wasserstein distances between D pairs of diagrams already on the device, and their gradient: the batched form
 * of Knowledge_Distillation/wasserstein.py (gudhi's wasserstein_distance(X, Y, order=q, internal_p=p,
 * enable_autodiff=True), :93, :198), PDGNN's training loss.  Pair t is X = points poff_x[t] .. poff_x[t+1] of
 * birth_x / death_x and Y = points poff_y[t] .. poff_y[t+1] of birth_y / death_y, in the batch imager's ragged layout:
 * poff[0] need not be 0, poff must be non-decreasing with entries in [0, Px] (resp. Py), a decreasing segment is empty.
 * kind_x / kind_y (either may be NULL: every point of that side counts) select the points whose kind k is < 32 with
 * bit k of kind_mask set.  q = order >= 1 finite, p = internal_p >= 1 or +inf.
 *   ground cost ||x - y||_p; distance of a point to the diagonal delta(x) = |d - b| * 2^(1/p - 1) (|d - b| / 2 for
 *   p = inf; the absolute value keeps PD_down and [max,min] points, which lie below the diagonal, at their distance);
 *   dist[t] = (sum c)^(1/q) minimised over partial matchings, c = ||x - y||_p^q for a matched pair and delta^q for a
 *   point matched to the diagonal -- gudhi's (n+1) x (m+1) transport problem, solved exactly (a shortest-augmenting-path
 *   assignment solver per pair, every loop bounded by the pair's point count).  Points with b == d go to the diagonal.
 *   A pair with a selected non-finite coordinate is not solved: dist NaN, all its matches -1.
 *   match_x[k] = the global index into the Y arrays of the point matched to X point k, -1 the diagonal, -2 a point
 *   masked out; match_y likewise from the Y side.  Both are written for every k in [poff[0], poff[D]) and nowhere else;
 *   either may be NULL.  A pair's matching and distance are the same bits from call to call and whatever the batch.
 * Workspace: dev_workspace of at least tlc_wasserstein_workspace_bytes(D, Px, Py) bytes (64 (Px + Py); Px, Py: the
 * lengths of the X and Y point arrays), 16-byte aligned; pair t uses the slice at 64 ((poff_x[t] - poff_x[0]) +
 * (poff_y[t] - poff_y[0])).  Neither call allocates or synchronises: both only enqueue on `stream`.
 * Gradient: with S = dist^q and G = grad_out[t], a point's gradient is G (1/q) S^(1/q - 1) dc/d(b, d) of the term it
 * appears in (the forward's matching), with torch.linalg.vector_norm's conventions: 0 for a zero-length difference,
 * sgn(0) = 0, ties of the p = inf max share the gradient evenly, S = 0 gives 0; NaN for the selected points of an
 * unsolved pair; 0 for masked points.  Written for every k in [poff[0], poff[D]) and nowhere else; any of the four
 * gradient pointers may be NULL.
 * TLC_E_INVALID: D outside [0, 2^31), Px or Py outside [0, 2^56), q < 1 or not finite, p < 1 or NaN, a NULL required
 * pointer with D > 0, or a workspace smaller than the query's size.  D = 0 with NULL pointers returns 0. */
int tlc_wasserstein_workspace_bytes(int64_t D, int64_t Px, int64_t Py, uint64_t *bytes);
int tlc_wasserstein_batch_dev(int device, int64_t D, int64_t Px, int64_t Py, const int64_t *dev_poff_x,
                              const double *dev_birth_x, const double *dev_death_x, const uint8_t *dev_kind_x,
                              const int64_t *dev_poff_y, const double *dev_birth_y, const double *dev_death_y,
                              const uint8_t *dev_kind_y, uint32_t kind_mask, double order, double internal_p,
                              void *dev_workspace, uint64_t workspace_bytes, double *dev_dist, int64_t *dev_match_x,
                              int64_t *dev_match_y, void *stream);
int tlc_wasserstein_batch_grad_dev(int device, int64_t D, const int64_t *dev_poff_x, const double *dev_birth_x,
                                   const double *dev_death_x, const uint8_t *dev_kind_x, const int64_t *dev_poff_y,
                                   const double *dev_birth_y, const double *dev_death_y, const uint8_t *dev_kind_y,
                                   uint32_t kind_mask, double order, double internal_p, const double *dev_dist,
                                   const int64_t *dev_match_x, const int64_t *dev_match_y, const double *dev_grad_out,
                                   double *dev_grad_birth_x, double *dev_grad_death_x, double *dev_grad_birth_y,
                                   double *dev_grad_death_y, void *stream);

/* Persistence diagrams of a batch of CALLER-SUPPLIED graphs under a filtration already on the device, and their gradient
 * in that filtration: Union_find + Accelerate_PD (accelerated_PD.py:26,115) per graph, batched -- the step in front of the
 * batch imager and the Wasserstein distances for a learnable filtration (Knowledge_Distillation/ConvCurv_GIN.py,
 * mode='filtration') or whole-graph persistence over a dataloader batch (Knowledge_Distillation/data_utils_GC.py:95-167).
 * The structure is uploaded and checked once; only f changes from call to call.
 *
 * tlc_graph_batch_create: D graphs; graph t owns vertices noff[t] .. noff[t+1] and edges eoff[t] .. eoff[t+1] of (ea, eb),
 * batch-global vertex ids (PyG's Batch.ptr / edge_index numbering).  HOST pointers, copied to `device`.  The order of a
 * graph's edges is the tie-break of the sweeps, as in tlc_union_find.  TLC_E_INVALID, with a message naming the first
 * offending graph or edge, unless noff and eoff start at 0 and are monotone, noff[D] < 2^31 and eoff[D] < 2^31, every edge
 * of graph t has both endpoints in [noff[t], noff[t+1]), no edge is a self-loop and no undirected edge appears twice (in
 * either direction).  Vertices without edges are allowed.  The call plans every graph's route from its size and allocates
 * every device buffer the diagram and gradient calls need: those never allocate.
 * tlc_graph_batch_pair_bound: N + M + D (N = noff[D], M = eoff[D]), the pair capacity every diagram call needs.
 *
 * tlc_graph_batch_diagrams_dev: dev_f float64[N].  Graph t's pairs and status are exactly what the pipeline gives for a
 * node-mode vicinity equal to that graph with filtration values f[noff[t] .. noff[t+1]] (tlc_vicinity_diagrams): PD_up,
 * [min,max], PD_down, [max,min], then PD_one with TLC_F_EXTENDED, birth / death values bit for bit, bv / dv batch-global
 * vertex ids; status DISCONNECTED (no pairs: no per-component diagrams), NO_TREE_EDGES (one vertex with TLC_F_EXTENDED,
 * keeps its 0-dim pairs), EMPTY (n = 0), and TLC_ST_NONFINITE (no pairs) for a graph with a NaN or +-inf value.  No
 * normalisation: the caller scales f (in torch, where it stays differentiable).  out->cap >= the pair bound; out->poff
 * [D+1] receives the exclusive offsets of the graphs' segments, compact and in graph order (poff[D] = pairs in total);
 * out->npairs [D] (may be NULL); kind / bv / dv / birth / death [cap] (each may be NULL: not written; entries past poff[D]
 * are left as they are); dev_status uint8[D] (may be NULL).  flags: TLC_F_EXTENDED, TLC_F_KEEP_ZERO, TLC_F_ASC_ONLY (not
 * with TLC_F_EXTENDED), TLC_F_NO_SMALL (every graph through the staged kernels 2 + 3 + 3b instead of kernel 9's fused
 * per-graph teams, which take graphs of <= 1024 vertices / <= 4096 edges; same results bit for bit).  Output is bit-identical
 * from call to call and independent of the rest of the batch.
 *
 * tlc_graph_batch_grad_dev: for the diagrams d of the last diagram call (device pointers: poff, bv, dv required),
 * grad_f[v] = sum over points k in [poff[0], poff[D]) with bv[k] == v of grad_birth[k] + with dv[k] == v of grad_death[k],
 * added in increasing k, birth term before death term, starting from 0.0; every v in [0, N) is written.  grad_birth /
 * grad_death may each be NULL (treated as 0).  Bit-reproducible: no floating-point atomics.
 *
 * All pointers of the two calls are DEVICE pointers on the batch's device; `stream` is a cudaStream_t (NULL: the legacy
 * default stream).  Both only enqueue (no synchronisation, no allocation, no host<->device traffic) and share the batch's
 * scratch: calls on one batch must be ordered (one stream, or the caller's events).  TLC_E_INVALID (bad flags, a NULL
 * required pointer) and TLC_E_CAPACITY (cap < bound) are returned before any CUDA call. */
typedef struct tlc_graph_batch tlc_graph_batch;
int tlc_graph_batch_create(int device, int64_t D, const int64_t *noff, const int64_t *eoff, const int32_t *ea,
                           const int32_t *eb, tlc_graph_batch **out);
int tlc_graph_batch_destroy(tlc_graph_batch *b);
int tlc_graph_batch_pair_bound(const tlc_graph_batch *b, int64_t *bound);
int tlc_graph_batch_diagrams_dev(tlc_graph_batch *b, const double *dev_f, uint32_t flags, tlc_diagrams *out,
                                 uint8_t *dev_status, void *stream);
int tlc_graph_batch_grad_dev(tlc_graph_batch *b, const tlc_diagrams *d, const double *dev_grad_birth,
                             const double *dev_grad_death, double *dev_grad_f, void *stream);

/* Hand-off of the cached image table to the decoder (baselines/TLCGNN.py:35-53): the table float64[rows][r2]
 * (the .npy cache layout, loaddatas.py:62-64,102) stays resident in HBM; out[i][:] = (float) table[row(i)][:],
 * row(i) = dev_index ? dev_index[i] : start + i -- what `torch.Tensor(PI[...]).cuda()` yields per decode call
 * on the host.  All pointers are DEVICE pointers on `device`; `stream` is a cudaStream_t (NULL: default
 * stream).  An index outside [0, rows) (numpy: IndexError) -> TLC_E_INVALID, the row is zero-filled. */
int tlc_pi_gather(int device, const double *dev_table, int64_t rows, int32_t r2, const int64_t *dev_index,
                  int64_t start, int64_t n, float *dev_out_f32, void *stream);

/* ---- multi-GPU: the exchange of the image rows as PEER STORES (SURVEY.md 8e; BASELINE.json north_star kernel 5) ----
 * The target list is sharded over the ranks of one node (one process per GPU, the CSR replicated); every rank needs the
 * whole table float32[rows][r2 + 1] afterwards (r2 image floats + the status as a float).  Instead of padding the shards
 * and calling an all-gather, every rank owns such a table and maps the tables of its peers through CUDA IPC; after the
 * shard's rows are computed, ONE kernel stores each row at its FINAL index into the table of every rank (remote ones over
 * NVLink / NVSwitch) and signals an arrival counter in each table; a one-thread kernel on the same stream then waits
 * until all ranks have arrived.  No host synchronisation, no NCCL, no un-permute pass.
 *   tlc_table_create : allocate this rank's table (zeroed); dev_rows receives the device address of row 0, handle64 the
 *                      64-byte CUDA IPC handle the host framework passes to the other ranks (any transport)
 *   tlc_table_attach : the handles of ALL ranks, ordered by rank ([nranks][64]); maps the peers' tables
 *   tlc_vicinity_pi_exchange : this rank's shard dev_targets[E][2] with the final row of each target dev_row_index[E]
 *                      (device buffers): tlc_vicinity_pi_dev + the exchange, asynchronous on the graph's stream; every
 *                      rank of the node must call it once per step (a rank with an empty shard passes E = 0)
 * Work queued behind the call on the graph's stream sees the complete table.  At most 16 ranks. */
int tlc_table_create(tlc_graph *g, int64_t rows, int32_t r2, void **dev_rows, unsigned char *handle64);
int tlc_table_attach(tlc_graph *g, int32_t nranks, int32_t my_rank, const unsigned char *handles64);
int tlc_vicinity_pi_exchange(tlc_graph *g, const int32_t *dev_targets, const int64_t *dev_row_index, int64_t E,
                             const tlc_params *p, int64_t *cnt_compute);

/* diffusion time of TLC_F_FILT_HKS (hks_time of data_utils_NC.compute_persistence_image, default 0.1); 0 < t <= 50 */
int tlc_graph_set_hks_time(tlc_graph *g, double t);

/* run this graph's kernels on a caller-owned CUDA stream (cudaStream_t as void*; NULL restores the
 * graph's own non-blocking stream -- to run on the legacy default stream pass cudaStreamLegacy, (void*)0x1).
 * Lets a host framework order the work with its own (e.g. NCCL) operations: buffers handed to
 * tlc_vicinity_pi_dev are written on this stream. */
int tlc_graph_set_stream(tlc_graph *g, void *stream);

/* introspection */
const char *tlc_last_error(void);
const char *tlc_version(void);
/* kernels launched by this library since load (the bench's gpu_launches counter) */
int64_t tlc_launch_count(void);
/* per-stage device time of the last tlc_vicinity_pi* call on this graph, ms, summed over chunks:
 * out[0..9] = sizes, fill, filtration, vertex order (2v), vertex-ordered sweep (3v), edge sort (2),
 * edge-sorted union-find (3), loops (3b), image (4), total; returns #chunks.
 * Only measured when the environment variable TLC_STAGE_TIMING=1 (adds event records). */
int tlc_last_stage_ms(tlc_graph *g, double *out10);
/* algorithmic bytes (SURVEY.md 8d: compulsory bytes B_e) summed over the targets of the last call */
int tlc_last_algorithmic_bytes(tlc_graph *g, double *bytes_total, double *bytes_bfs, double *bytes_uf);

/* totals over the live targets of the last call: out[0] = live targets, out[1] = sum n, out[2] = sum m,
 * out[3] = chunks, out[4] = targets the vertex-ordered sweep handed back to the edge-sorted kernels,
 * out[5..7] = blocks of the vertex order through the general path / the row check / in total (kernel 3v) */
int tlc_last_counts(tlc_graph *g, int64_t *out8);
/* targets of the last call that took the graph-row route (TLC_F_DIRECT / TLC_F_NO_DIRECT) */
int64_t tlc_last_direct(tlc_graph *g);
/* targets of the last call whose filtration came from the per-root shortest-path tables (kernel 1t; TLC_F_NO_TABLE).  For
 * those targets of a BATCH call the induced edges are not counted (no kernel reads all their rows any more): they are
 * missing from tlc_last_counts' sum m and from the 16 m term of tlc_last_algorithmic_bytes; tlc_vicinity_sizes counts them. */
int64_t tlc_last_table(tlc_graph *g);
/* of those, the targets kernel 1t ran with both roots u and v in the same passes (their two states fit its shared memory;
 * TLC_TABLE_ONE_ROOT=1 runs every target one root at a time) */
int64_t tlc_last_table_two_root(tlc_graph *g);
/* device ms the one-time build of the shortest-path tables took (all N roots, at the first graph-row call that uses them) */
double tlc_table_build_ms(tlc_graph *g);
/* kernel S in the last call: out[0..2] = device ms of the class A (warp per target, n <= 64) / class B (128-thread CTA,
 * n <= 256) / class C (256-thread CTA, n <= 1024) launch (TLC_STAGE_TIMING=1), out[3..5] = rows they finished,
 * out[6] = rows handed on to the staged pipeline */
int tlc_last_small(tlc_graph *g, double *out7);

#ifdef __cplusplus
}
#endif
#endif
