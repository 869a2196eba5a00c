/* klu.h -- C ABI of the B200 lattice forward-backward / posterior-indexing engine.
 *
 * The reference (jpuigcerver/kaldi-lattice-utils) has no FFI: its boundary is the
 * per-lattice functor body of each command-line tool, between
 * `lattice_reader.Value()` and `writer.Write()`.  Every entry point below replaces
 * one of those bodies for a whole BATCH of lattices (file:line relative to
 * /root/reference):
 *
 *   KLU_SEGMENT        kwsbin2/lattice-word-index-segment.cc:31-72,134-177,96-128
 *   KLU_POSITION       kwsbin2/lattice-word-index-position.cc:33-76,135-190,100-129
 *                      (+ fstext/fstext-utils2.h:109-215)
 *   KLU_UTTERANCE      kwsbin2/lattice-word-index-utterance.cc:87-190,274-311
 *   KLU_FRAME_POST     latbin/lattice-to-word-frame-post.cc:68-140
 *   KLU_PRUNE_DYN_BEAM latbin/lattice-prune-dyn-beam.cc:27-90,148-207
 *   KLU_BEST_PATH2     latbin/lattice-best-path2.cc:78-211
 *                      (+ fstext/fstext-utils2.h:109-271)
 *   KLU_CHAR_POSITION  kwsbin2/lattice-char-index-position.cc:137-284
 *                      (+ kwsbin2/utils.h:41-303, fstext/fstext-utils2.h:278-603)
 *   KLU_POSITION_POST  latbin/lattice-to-word-position-post.cc:70-141 (SURVEY.md 8f)
 *   KLU_CHAR_SEGMENT   kwsbin2/lattice-char-index-segment.cc:93-223 (SURVEY.md 8f)
 *                      (both char tools: the pseudo-word frontier is bounded by --nbest, see
 *                      klu_opts.nbest)
 *   KLU_LENGTH_DIST    latbin/lattice-to-transcript-length-dist.cc:64-125 (SURVEY.md 8f)
 *   KLU_PRUNE_ARCS     latbin/lattice-prune-arcs.cc:34-84,136-165 (SURVEY.md 8f)
 *
 * Plain pointers and sizes only; all pointers are HOST pointers.  Every function
 * returns 0 on success; on failure klu_last_error() (thread-local) explains.
 * There is no CPU fallback: klu_create() fails when no CUDA device is usable.
 *
 * Lattice layout handed to klu_load() (one CompactLattice = one "lattice"):
 *   states are numbered topologically (every arc has src < dst) with start == 0
 *   (what TopSortCompactLatticeIfNeeded guarantees; klu_topsort() does it on the
 *   host when needed); arcs are grouped by ascending src in stored order
 *   (OpenFst's state/arc iteration order); arc duration = length of the
 *   transition-id string on the arc; a non-final state has final weight
 *   (+inf,+inf) (LatticeWeight::Zero()).
 */
#ifndef KLU_H_
#define KLU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KLU_VERSION 3

typedef struct klu_ctx klu_ctx; /* one per GPU; owns a stream and all device buffers */

enum klu_tool {
  KLU_SEGMENT = 0,
  KLU_POSITION = 1,
  KLU_UTTERANCE = 2,
  KLU_FRAME_POST = 3,
  KLU_PRUNE_DYN_BEAM = 4,
  KLU_BEST_PATH2 = 5,
  KLU_CHAR_POSITION = 6,
  KLU_FWD_BWD = 7, /* alpha/beta only (ComputeLatticeAlphasAndBetas [ext]) */
  KLU_POSITION_POST = 8,
  KLU_CHAR_SEGMENT = 9,
  KLU_LENGTH_DIST = 10,
  KLU_PRUNE_ARCS = 11
};

/* A batch of lattices as concatenated SoA arrays.  state_off/arc_off have
 * num_lattices+1 entries; arc_src/arc_dst are lattice-LOCAL state ids. */
typedef struct klu_lattices {
  int32_t num_lattices;
  const int64_t* state_off;
  const int64_t* arc_off;
  const int32_t* arc_src;
  const int32_t* arc_dst;
  const int32_t* arc_label;
  const int32_t* arc_dur;
  const float* arc_graph;
  const float* arc_acoustic;
  const float* fin_graph;    /* per state; +inf = not final */
  const float* fin_acoustic; /* per state; +inf = not final */
  const int32_t* fin_dur;    /* per state; may be NULL (all 0) */
  /* Optional: arcs leaving each state (fst NumArcs(s)), concatenated like fin_graph.  When
   * given, arc_src may be NULL -- the arcs of a lattice are then taken to be grouped by
   * source state in state order (how OpenFst stores them), which saves a sixth of the
   * host-to-device traffic. */
  const int32_t* state_num_arcs;
  /* Optional compact forms; each replaces its 32-bit array (which may then be NULL) and cuts the
   * host-to-device traffic: durations that all fit a byte, and destinations as dst - src when
   * every difference fits 16 bits (a topologically sorted lattice has dst > src).  20 -> 15 bytes
   * per arc together with state_num_arcs. */
  const uint8_t* arc_dur_u8;
  const uint16_t* arc_dst_delta_u16;
  /* Labels that all fit 16 bits (a vocabulary below 65536 words): replaces arc_label, 15 -> 13
   * bytes per arc. */
  const uint16_t* arc_label_u16;
} klu_lattices;

/* Command-line flags of the tools (SURVEY.md 8b).  klu_opts_default() fills the
 * reference defaults. */
typedef struct klu_opts {
  float acoustic_scale;    /* --acoustic-scale   1.0 */
  float graph_scale;       /* --graph-scale      1.0 */
  float insertion_penalty; /* --insertion-penalty 0.0 */
  float beam;              /* --beam             +inf (index tools only) */
  const int32_t* include_words; /* --include-words (wins over exclude when non-empty) */
  int32_t num_include;
  const int32_t* exclude_words; /* --exclude-words */
  int32_t num_exclude;
  float beam_ratio;   /* --beam-ratio 0.9   (prune-dyn-beam) */
  float min_beam;     /* --min-beam   1e-3  (prune-dyn-beam) */
  int32_t max_arcs;   /* --max-arcs   INT_MAX */
  int32_t max_states; /* --max-states INT_MAX */
  int32_t nbest;      /* --nbest 100 (char index).  Also bounds the work: a pseudo-word prefix
                       * none of whose extensions can still reach a lattice's nbest best rows is
                       * not expanded (an exact cut: the rows and their order are those of the
                       * uncut search).  A lattice fails with "more than 2^24 trie nodes at one
                       * depth" only when nbest is not below its row count and its uncut frontier
                       * is that large. */
  /* char index label groups (kwsbin2/utils.h:41-84): parallel arrays label->group
   * (epsilon->0 and whitespace->1 included by the caller), the groups that
   * increment the word count (INT_MAX = default group, 2, 3, ...), and the
   * deleted groups ({1}). */
  const int32_t* group_labels;
  const int32_t* group_ids;
  int32_t num_group_labels;
  const int32_t* inc_groups;
  int32_t num_inc_groups;
  const int32_t* del_groups;
  int32_t num_del_groups;
} klu_opts;

const char* klu_last_error(void);
int klu_version(void);
void klu_opts_default(klu_opts* o);

int klu_device_count(int* n);
int klu_create(int device, klu_ctx** out);
int klu_destroy(klu_ctx* ctx);

/* Pinned host memory (callers that parse arks straight into pinned buffers get
 * asynchronous H2D without a staging copy). */
int klu_host_alloc(size_t bytes, void** out);
int klu_host_free(void* p);

/* Host-side helper mirroring TopSortCompactLatticeIfNeeded [ext]: renumbers ONE
 * lattice in place when some arc has src >= dst (OpenFst TopSort order: reverse
 * DFS finishing order from the start state) and regroups arcs by new src.
 * order_out (nstates, may be NULL) receives new id of each old state.  Returns
 * non-zero on a cyclic lattice. */
int klu_topsort(int32_t nstates, int64_t narcs, int32_t* arc_src, int32_t* arc_dst, int32_t* arc_label,
                int32_t* arc_dur, float* arc_graph, float* arc_acoustic, float* fin_graph, float* fin_acoustic,
                int32_t* fin_dur, int32_t* order_out);

/* Packer + H2D: level-buckets and uploads the batch (replaces the current one). */
int klu_load(klu_ctx* ctx, const klu_lattices* lats);

/* Runs one tool over the loaded batch; asynchronous on the context's stream.
 * Results stay in device memory until fetched. */
int klu_run(klu_ctx* ctx, int tool, const klu_opts* opts);
int klu_sync(klu_ctx* ctx);

/* ---- results (each call synchronises the stream first) ----------------------
 * Entry tables: klu_result_offsets() gives entry_off[num_lattices+1]; the fetch
 * calls fill arrays of entry_off[num_lattices] elements, lattice after lattice
 * in INPUT order, each lattice's entries in the reference's output order. */
int klu_result_offsets(klu_ctx* ctx, int64_t* entry_off);
int klu_fetch_segment(klu_ctx* ctx, int32_t* word, int32_t* t0, int32_t* t1, double* logp);
int klu_fetch_position(klu_ctx* ctx, int32_t* word, int32_t* pos, int32_t* t0, int32_t* t1, double* logp);
int klu_fetch_utterance(klu_ctx* ctx, int32_t* word, double* logp);
/* frame-post: num_frames[num_lattices] (Posterior length incl. empty frames);
 * entries carry their frame index. */
int klu_fetch_frame_post(klu_ctx* ctx, int32_t* num_frames, int32_t* frame, int32_t* word, float* logp);
/* The same rows without the per-row frame column (a third of the download): frame_row_off has
 * num_frames[l] + 1 entries per lattice, lattice after lattice; entry k of lattice l is the first
 * row of frame k counted from the lattice's first row (klu_result_offsets), the last entry the
 * lattice's row count -- the shape of the Posterior the reference writes
 * (latbin/lattice-to-word-frame-post.cc:106-128: one vector of (word, post) pairs per frame). */
int klu_fetch_frame_post_csr(klu_ctx* ctx, int32_t* num_frames, int64_t* frame_row_off, int32_t* word, float* logp);
/* position-post: num_positions[num_lattices] (Posterior length = longest label sequence);
 * entries carry their 0-based position index. */
int klu_fetch_position_post(klu_ctx* ctx, int32_t* num_positions, int32_t* position, int32_t* word, float* logp);
/* length-dist: entries are (transcript length, float log-posterior), one Posterior frame per lattice. */
int klu_fetch_length_dist(klu_ctx* ctx, int32_t* length, float* logp);
/* best-path2: entries are the transcript labels; cost[num_lattices] (float path
 * cost, latbin/lattice-best-path2.cc:192), num_frames[num_lattices]. */
int klu_fetch_best_path2(klu_ctx* ctx, int32_t* label, float* cost, int32_t* num_frames);
/* prune-dyn-beam and prune-arcs (for the latter beams[2*l] = beam - total, [2*l+1] = rank of
 * the first arc put back; a state's arcs come in the order AddArc left them): entries are surviving arcs: index of the arc in the caller's
 * arrays (lattice-local), its new src/dst state ids and its output weights
 * (original scale after the float round trip, :188-192).  state_map has one
 * entry per input state (concatenated like fin_graph): new id or -1; fin_* are
 * per input state output final weights.  beams[2*l] = original beam, [2*l+1] =
 * final beam. */
int klu_fetch_prune(klu_ctx* ctx, int32_t* arc_index, int32_t* new_src, int32_t* new_dst, float* graph,
                    float* acoustic, int32_t* state_map, float* fin_graph, float* fin_acoustic, double* beams);
/* char index: per entry the pseudo-word is chars[char_off[i] .. char_off[i+1])
 * (labels to be joined with '_').  Call klu_result_char_sizes() first. */
int klu_result_char_sizes(klu_ctx* ctx, int64_t* total_chars);
int klu_fetch_char_position(klu_ctx* ctx, int64_t* char_off, int32_t* chars, int32_t* pos, int32_t* t0,
                            int32_t* t1, double* logp);
/* char segment index (KLU_CHAR_SEGMENT): same layout, rows carry (t0, t1) only. */
int klu_fetch_char_segment(klu_ctx* ctx, int64_t* char_off, int32_t* chars, int32_t* t0, int32_t* t1, double* logp);
/* KLU_FWD_BWD / any run: per-state alpha, beta (input state numbering) and
 * per-lattice total = 0.5*(tot_fwd + beta[0]) */
int klu_fetch_fwd_bwd(klu_ctx* ctx, double* alpha, double* beta, double* total);

/* ---- measurement -----------------------------------------------------------*/
/* CUDA-event timer on the context's stream. */
int klu_timer_start(klu_ctx* ctx);
int klu_timer_stop(klu_ctx* ctx, float* ms);
/* Kernel launches issued by this context so far. */
int klu_launch_count(klu_ctx* ctx, int64_t* n);
/* Per-kernel CUDA-event profile: enable, run, then read a JSON object
 * {"kernel": {"launches": n, "ms": total}, ...} into buf. */
int klu_profile_enable(klu_ctx* ctx, int on);
int klu_profile_json(klu_ctx* ctx, char* buf, size_t cap);
/* Device-side cost of the last klu_load, for honest throughput figures: upload_ms = wall
 * clock of the host-to-device copies of the caller's arrays; pack_ms = CUDA-event time of
 * the device packer (levels, CSR, bands); frame_index_ms = CUDA-event time of the per-batch
 * indexes built on first use: the frame index of the first KLU_FRAME_POST run on the batch, the
 * start-frame buckets of the first KLU_SEGMENT run (0 until then). */
int klu_load_times(klu_ctx* ctx, float* upload_ms, float* pack_ms, float* frame_index_ms);
/* Totals of the loaded batch: {lattices, states, arcs, levels, entries of last run}. */
int klu_batch_stats(klu_ctx* ctx, int64_t stats[8]);
/* Writes `bytes` of device memory to evict L2 between timed iterations. */
int klu_flush_l2(klu_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* KLU_H_ */
