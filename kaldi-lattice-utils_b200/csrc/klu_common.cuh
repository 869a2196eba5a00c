// klu_common.cuh -- shared declarations of the B200 lattice engine (internal).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <time.h>

#include <map>
#include <string>
#include <vector>

#include "klu.h"

namespace klu {

void set_error(const std::string& msg);

#define KLU_CUDA(call)                                                                      \
  do {                                                                                      \
    cudaError_t err__ = (call);                                                             \
    if (err__ != cudaSuccess) {                                                             \
      klu::set_error(std::string(#call) + ": " + cudaGetErrorString(err__) + " at " + __FILE__ + ":" + \
                     std::to_string(__LINE__));                                             \
      return 1;                                                                             \
    }                                                                                       \
  } while (0)

#define KLU_TRY(call)            \
  do {                           \
    int rc__ = (call);           \
    if (rc__ != 0) return rc__;  \
  } while (0)

// Growable device buffer, reused across runs (no cudaMalloc in steady state).
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);
  void release();
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// KLU_TRACE=1: wall-clock marks of the host-side phases on stderr (pipelining diagnostics).
inline void klu_trace(const void* c, const char* what) {
  static const bool on = getenv("KLU_TRACE") != nullptr;
  if (!on) return;
  timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  fprintf(stderr, "[klu %p] %.3f %s\n", c, ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6, what);
}

// The packer's metadata transfers (per-lattice arrays, KBs) do not use the copy engines:
// those are shared by all contexts of the device, and a small copy queued behind another
// context's multi-hundred-MB upload or result download waits for all of it -- with the
// packing kernels of this context behind it.  They go through a pinned staging area
// instead, which a one-line kernel reads or writes over PCIe directly.
//   small_h2d: stream-ordered copy of `bytes` (multiple of 4) to the device; src may be reused at return.
//   small_d2h: queues a read; dst_host is filled by the next small_sync().
//   small_sync: cudaStreamSynchronize + delivery of the queued reads.
// stage_begin() (start of klu_load) sizes the area for L lattices and recycles it.
int stage_begin(klu_ctx* c, size_t L);
int small_h2d(klu_ctx* c, void* dst_dev, const void* src_host, size_t bytes);
int small_d2h(klu_ctx* c, void* dst_host, const void* src_dev, size_t bytes);
int small_sync(klu_ctx* c);

// How arc/final weights become costs (SURVEY.md 8a P2, P3, P6, P7, F1).
struct CostParams {
  double gs, as;   // graph / acoustic scale (double products, float storage)
  float gsf, asf;  // the same scales as the floats the flags are (gs == (double)gsf)
  float pen;       // insertion penalty (float add on arcs with label != 0)
  int scale;       // apply gs/as (either != 1)
  int float_sum;   // cost = (double)(float)(g + a) instead of (double)g + (double)a
};

// Packed batch, device side.  States are renumbered per lattice by (level, input
// id); "level" = longest arc distance from any source state, so all arcs into a
// level come from earlier levels and a level is a contiguous state range.
struct BatchView {
  int32_t L;          // lattices
  int32_t S;          // states
  int32_t E;          // arcs
  const int32_t* s_off;      // [L+1] first state of each lattice
  const int32_t* e_off;      // [L+1] first arc of each lattice
  const int32_t* lvl_off;    // [L+1] index into lvl_start (each lattice has nl+1 entries)
  const int32_t* lvl_start;  // first (global) state of each level, + sentinel per lattice
  const int4* in_rec;        // [E] arcs sorted by dst: {src(global), g bits, a bits, label}
  const int4* out_rec;       // [E] arcs sorted by src: {dst(global), g bits, a bits, label}
  const int32_t* in_off;     // [S+1]
  const int32_t* out_off;    // [S+1]
  const int32_t* out_src;    // [E] (global) src of out-order arcs
  const int32_t* out_orig;   // [E] lattice-local index of the arc in the caller's arrays
  const int32_t* in2out;     // [E] position (global) of each in-order arc in the out-order arrays
  const float* fin_g;        // [S]
  const float* fin_a;        // [S]
  const int32_t* time;       // [S] frame of each state (CompactLatticeStateTimes)
  const int32_t* orig;       // [S] lattice-local input id of each state
  const int32_t* old2new;    // [S] input state (global) -> packed state (global)
  const int32_t* level;      // [S] level index of each state within its lattice
  const int32_t* band_lo;    // [S] min #non-eps labels on paths from the start (-1: unreachable)
  const int64_t* band_off;   // [S+1] offsets into the (state,len) band arrays
  const int32_t* order;      // [L] lattices by descending arc count (work queue order)
  const int32_t* fr_base;    // [L+1] first slot of each lattice in fr_off (num_frames + 1 slots per lattice)
  const int64_t* fr_off;     // per (lattice, frame): first entry of the frame in frame_arc
  const int32_t* frame_arc;  // per frame: out-order arc ids (global) of the word arcs alive in it, sorted by
                             // (word, arc); bit 31 marks the first arc of every word group
};

struct KernelStat {
  int64_t launches = 0;
  double ms = 0;
};

}  // namespace klu

struct klu_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  // small_h2d / small_d2h: pinned staging area read / written by kernels (no copy engine)
  char* h_stage = nullptr;
  size_t stage_cap = 0, stage_used = 0;
  struct StagedRead {
    void* dst;
    size_t off, bytes;
  };
  std::vector<StagedRead> stage_reads;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_p0 = nullptr, ev_p1 = nullptr;  // around the device packer
  float load_upload_ms = 0.f, load_pack_ms = 0.f, lazy_pack_ms = 0.f;  // klu_load_times
  bool frame_ready = false;  // frame index of the loaded batch built (klu_frame.cu; on first use)
  bool seg_ready = false;    // arcs bucketed by start frame (klu_segment.cu; on first use)
  int32_t seg_max_bucket = 0, seg_slots = 0;
  int num_sms = 148;
  int64_t launches = 0;
  bool profile = false;
  std::map<std::string, klu::KernelStat> prof;
  std::vector<std::pair<std::string, std::pair<cudaEvent_t, cudaEvent_t> > > prof_pending;
  std::vector<cudaEvent_t> event_pool;

  // ---- loaded batch (host metadata) ----
  bool loaded = false;
  int32_t L = 0;
  int64_t S = 0, E = 0, NL = 0;
  std::vector<int64_t> h_s_off, h_e_off;     // input offsets
  std::vector<int32_t> h_new2old;            // per packed state: input local id
  std::vector<int32_t> h_old2new;            // per input state (global): packed global id
  std::vector<int32_t> h_num_frames;         // utterance length per lattice
  std::vector<int32_t> h_maxtime;            // largest state time per lattice
  std::vector<uint8_t> h_times_ok;           // consistent state times per lattice
  std::vector<int64_t> h_cap_frame, h_cap_pos;  // per lattice entry upper bounds
  std::vector<int32_t> h_maxlen;             // max #non-eps labels on a path, per lattice
  std::vector<int64_t> h_band_off;           // [L+1] first band cell of each lattice
  std::vector<int32_t> h_fr_base;            // [L+1] frame slots
  int64_t frame_entries = 0;                 // sum over lattices of arc x frame instances
  std::vector<int64_t> h_frame_res_off;      // [L+1] frame-post output rows per lattice (static per batch)
  int32_t fr_items = 0;                      // frame-post work items (runs of frames)
  int32_t fr_max_window = 0;                 // largest arc window of a run of frames
  int32_t max_label = 0, max_time = 0, max_len = 0, max_indeg = 0, max_outdeg = 0, max_states = 0;
  int32_t max_span = 0;  // longest arc in frames (time[dst] - time[src])
  double avg_deg = 0;
  int64_t band_total = 0;

  // ---- device: packed batch ----
  klu::DevBuf d_s_off, d_e_off, d_lvl_off, d_lvl_start, d_in_rec, d_out_rec, d_in_off, d_out_off, d_out_src,
      d_in2out, d_old2new, d_out_orig, d_fin_g, d_fin_a, d_time, d_orig, d_level, d_band_lo, d_band_off, d_order, d_fr_base, d_fr_off, d_frame_arc,
      d_fr_item, d_fr_gloc, d_fr_res_off, d_fr_gword, d_fr_gstart, d_fr_gframe, d_fr_run_lo, d_fr_run_hi, d_fr_tarc, d_fr_tlabel, d_fr_seg, d_tile_heads, d_sg_meta, d_sg_boff, d_sg_perm, d_sortws;
  // ---- device: per-run state ----
  klu::DevBuf d_alpha, d_beta, d_total, d_totfwd, d_counter, d_filter;
  klu::DevBuf d_vfwd, d_vbwd, d_best;  // tropical sweeps
  klu::DevBuf d_alpha2;                // banded alpha[s][len]
  klu::DevBuf d_scratch[12];           // tool scratch (keys, indices, values ...)
  klu::DevBuf d_res[8];                // dense results of the last run
  klu::DevBuf d_flush;
  klu::DevBuf d_char[80];              // frontier / trie / row buffers of the character tools (klu_char.cu)

  // ---- last run ----
  int last_tool = -1;
  std::vector<int64_t> h_res_off;  // [L+1] entries per lattice of the last run
  int64_t last_entries = 0;
  int64_t last_chars = 0;
  bool frame_col_static = false;  // last frame-post run used the static frame column
  void* char_state = nullptr;  // host-side rows of the last char-index run (klu_char.cu)

  klu::BatchView view() const;
};

namespace klu {

// Launch bookkeeping: counts launches and (when profiling) brackets the launch
// with CUDA events on the context's stream.
struct LaunchScope {
  klu_ctx* c;
  const char* name;
  cudaEvent_t a = nullptr, b = nullptr;
  LaunchScope(klu_ctx* ctx, const char* n);
  ~LaunchScope();
};
#define KLU_LAUNCH(ctx, name) klu::LaunchScope scope__(ctx, name)

int check_launch(const char* what);

// klu_pack.cu
int pack_and_upload(klu_ctx* c, const klu_lattices* lats);       // host packer (KLU_HOST_PACKER=1)
// klu_gpack.cu
int pack_and_upload_gpu(klu_ctx* c, const klu_lattices* lats);   // device packer (default)
int ensure_frame_index(klu_ctx* c);  // frame -> arc offsets + (frame, word) groups, on first use
// klu_sweep.cu
int run_log_sweeps(klu_ctx* c, const CostParams& cp, bool use_beam, float beam);
int run_tropical_sweeps(klu_ctx* c, const CostParams& cp);
int run_banded_alpha(klu_ctx* c, const CostParams& cp, bool use_beam, float beam, int l0, int l1);
// klu_index.cu
int run_index_tool(klu_ctx* c, int tool, const klu_opts* o);
// klu_segment.cu: lattice-word-index-segment by start-frame buckets; *done = false -> use run_index_tool
int run_segment_buckets(klu_ctx* c, const klu_opts* o, bool* done);
// klu_position.cu: lattice-word-index-position, lattice-to-word-position-post, lattice-best-path2
int run_position_tool(klu_ctx* c, int tool, const klu_opts* o);
// klu_frame.cu
int build_frame_groups(klu_ctx* c);  // pack time: (frame, word)-sorted instances, head bits, output offsets
int run_frame_post(klu_ctx* c, const klu_opts* o);
// klu_prune.cu
int run_prune_dyn_beam(klu_ctx* c, const klu_opts* o);
int run_prune_arcs(klu_ctx* c, const klu_opts* o);  // lattice-prune-arcs (SURVEY.md 8f rank 4)
// klu_bestpath.cu: decode stage of lattice-best-path2 for lattices [l0, l1); the
// (label, position) posteriors were already turned into per-entry float costs.
struct BestPathChunk {
  int l0, l1;
  long long band_base;            // first band cell of the chunk
  const double* alpha2;           // chunk-local banded alpha
  const long long* arc_cellbase;  // [E] per out-order arc: its (label, position) cell = arc_cellbase[e] + position
  const double* ecost;            // per (label, position) cell: (double)(float) cost 1 - P
  bool first_chunk;
};
int best_path2_decode(klu_ctx* c, const CostParams& cp, const BestPathChunk& ch);
// klu_lendist.cu
int run_length_dist(klu_ctx* c, const klu_opts* o);
// klu_char.cu
int run_char_position(klu_ctx* c, const klu_opts* o);
int run_char_segment(klu_ctx* c, const klu_opts* o);
void char_release(klu_ctx* c);

CostParams make_cost_params(const klu_opts* o, bool float_sum);
int pick_group(double avg_deg);  // lanes cooperating on one state, from the mean degree

#define KLU_DISPATCH_G(G, ...)                              \
  switch (G) {                                              \
    case 2: { constexpr int kG = 2; __VA_ARGS__; } break;   \
    case 4: { constexpr int kG = 4; __VA_ARGS__; } break;   \
    case 8: { constexpr int kG = 8; __VA_ARGS__; } break;   \
    case 16: { constexpr int kG = 16; __VA_ARGS__; } break; \
    default: { constexpr int kG = 32; __VA_ARGS__; } break; \
  }

int upload_filter(klu_ctx* c, const klu_opts* o, int* mode_out, int* n_out);

// klu_core.cu: per-lattice counts -> offsets by one CTA (launched and counted as `label`):
// off[l] = off[l0] + cnt[l0] + ... + cnt[l - 1] for l in (l0, l1].  With l0 > 0, off[l0] must hold
// the total of the lattices before l0 (a chunked run); with l0 == 0 the scan starts from 0 and
// does not read off[0].  off may be cnt itself (the packer's totals, scanned in place).
int scan_counts(klu_ctx* c, const int32_t* cnt, int l0, int l1, int64_t* off, const char* label);
int scan_counts(klu_ctx* c, const long long* cnt, int l0, int l1, long long* off, const char* label);

}  // namespace klu

// ---------------------------------------------------------------------------
// Device helpers
#ifdef __CUDACC__
namespace klu {

// Kernels launched on a (lattices, tiles) grid: CTAs are dispatched x-fastest, so with the lattice
// in blockIdx.x the ~1000 CTAs in flight touch ~1000 different lattices and their gathers (alpha,
// beta, entries by sorted index) miss L2.  lat_tile() re-reads the same grid tile-fastest: the
// CTAs in flight then cover a few lattices whose arrays stay in L2 (k_gather: 4.4 -> 0.9 ms).
struct LatTile {
  int l, tile, tiles;
};
__device__ __forceinline__ LatTile lat_tile() {
  const unsigned long long lin = (unsigned long long)blockIdx.y * gridDim.x + blockIdx.x;
  LatTile t;
  t.tiles = (int)gridDim.y;
  t.l = (int)(lin / gridDim.y);
  t.tile = (int)(lin % gridDim.y);
  return t;
}

__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }
__device__ __forceinline__ double pos_inf() { return __longlong_as_double(0x7ff0000000000000LL); }

// Arc cost exactly as the reference builds it: ScaleLattice (double product ->
// float), AddWordInsPenToCompactLattice (float add), then ConvertToCost (double
// sum) or the float sum of ComputeCompactLatticeBetas / word-frame-post.
__device__ __forceinline__ void scaled_weights(float g, float a, int label, const CostParams& cp, float* go,
                                               float* ao) {
  if (cp.scale && !(isinf(g) && isinf(a) && g > 0 && a > 0)) {
    g = (float)__dmul_rn(cp.gs, (double)g);
    a = (float)__dmul_rn(cp.as, (double)a);
  }
  if (label != 0) g = __fadd_rn(g, cp.pen);
  *go = g;
  *ao = a;
}

__device__ __forceinline__ double arc_cost(float g, float a, int label, const CostParams& cp) {
  float g2, a2;
  scaled_weights(g, a, label, cp, &g2, &a2);
  if (cp.float_sum) return (double)__fadd_rn(g2, a2);
  return __dadd_rn((double)g2, (double)a2);
}

// Cost of an arc record.  Arc weights are FINITE (klu_load rejects anything else).
// ScaleLattice forms (float)(scale * (double)w); the scale is a float-valued double,
// so that double product is exact (24 + 24 bits) and its rounding to float is the
// IEEE float product: one FMUL instead of F2F / DMUL / F2F.
__device__ __forceinline__ double rec_cost(const int4& r, const CostParams& cp) {
  float g = __int_as_float(r.y), a = __int_as_float(r.z);
  if (cp.scale) {
    g = __fmul_rn(cp.gsf, g);
    a = __fmul_rn(cp.asf, a);
  }
  if (r.w != 0) g = __fadd_rn(g, cp.pen);
  if (cp.float_sum) return (double)__fadd_rn(g, a);
  return __dadd_rn((double)g, (double)a);
}

// final weights: no insertion penalty (label 0)
__device__ __forceinline__ double final_cost(float g, float a, const CostParams& cp) {
  return arc_cost(g, a, 0, cp);
}

// [ext] kaldi LogAdd(double,double): max + log1p(exp(-|d|)), cut at log(DBL_EPSILON)
__device__ __forceinline__ double log_add(double x, double y) {
  double diff;
  if (x < y) {
    diff = x - y;
    x = y;
  } else {
    diff = y - x;
  }
  if (diff >= -36.04365338911715) return x + log1p(exp(diff));
  return x;
}

// ---- cheap f64 exp / log for the level sweeps -------------------------------
// Taylor coefficients 1/11! .. 1/3! and 2/17 .. 2/3, in constant memory so each DFMA
// takes its coefficient as a constant-bank operand.
static __constant__ double kExpPoly[9] = {1.0 / 39916800.0, 1.0 / 3628800.0, 1.0 / 362880.0, 1.0 / 40320.0, 1.0 / 5040.0,
                                   1.0 / 720.0,      1.0 / 120.0,     1.0 / 24.0,     1.0 / 6.0};
static __constant__ double kLogPoly[8] = {2.0 / 17.0, 2.0 / 15.0, 2.0 / 13.0, 2.0 / 11.0, 2.0 / 9.0, 2.0 / 7.0, 2.0 / 5.0, 2.0 / 3.0};

// exp(d) for the terms of a log-sum (relative error < 1e-14, checked on the host
// against libm over [-700, 700]): round-to-nearest range reduction with the
// 1.5 * 2^52 trick, degree-11 Taylor polynomial on |r| <= ln2/2, exponent patched
// in with an integer add.  d < -700 (and NaN) gives 0, d > 700 gives +inf.
__device__ __forceinline__ double fast_exp(double d) {
  if (!(fabs(d) <= 700.0)) return d < 0.0 ? 0.0 : pos_inf();  // NaN -> +inf (callers treat it as "redo exactly")
  const double t = __fma_rn(d, 1.4426950408889634, 6755399441055744.0);
  const int k = __double2loint(t);
  const double kf = __dadd_rn(t, -6755399441055744.0);
  double r = __fma_rn(kf, -6.93147180369123816490e-01, d);
  r = __fma_rn(kf, -1.90821492927058770002e-10, r);
  double p = kExpPoly[0];
  p = __fma_rn(p, r, kExpPoly[1]);
  p = __fma_rn(p, r, kExpPoly[2]);
  p = __fma_rn(p, r, kExpPoly[3]);
  p = __fma_rn(p, r, kExpPoly[4]);
  p = __fma_rn(p, r, kExpPoly[5]);
  p = __fma_rn(p, r, kExpPoly[6]);
  p = __fma_rn(p, r, kExpPoly[7]);
  p = __fma_rn(p, r, kExpPoly[8]);
  p = __fma_rn(p, r, 0.5);
  p = __fma_rn(p, r, 1.0);
  p = __fma_rn(p, r, 1.0);
  return __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));
}

// log(s) for a positive NORMAL double (callers check the range): s = 2^k * m with
// m in [sqrt(1/2), sqrt(2)), log m = 2 atanh((m-1)/(m+1)) as an odd series; the
// reciprocal comes from rcp.approx + two Newton steps.  Absolute error < 1e-15
// relative to max(1, |log s|) (host check).
__device__ __forceinline__ double fast_log(double s) {
  int hi = __double2hiint(s);
  int k = (hi >> 20) - 1023;
  hi = (hi & 0x000fffff) | 0x3ff00000;
  if (hi >= 0x3ff6a09f) {
    hi -= 0x00100000;
    ++k;
  }
  const double m = __hiloint2double(hi, __double2loint(s));
  const double den = __dadd_rn(m, 1.0), num = __dadd_rn(m, -1.0);
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(den));
  double e = __fma_rn(-den, y, 1.0);
  y = __fma_rn(y, e, y);
  e = __fma_rn(-den, y, 1.0);
  y = __fma_rn(y, e, y);
  double f = __dmul_rn(num, y);
  f = __fma_rn(__fma_rn(-den, f, num), y, f);
  const double f2 = __dmul_rn(f, f);
  double p = kLogPoly[0];
  p = __fma_rn(p, f2, kLogPoly[1]);
  p = __fma_rn(p, f2, kLogPoly[2]);
  p = __fma_rn(p, f2, kLogPoly[3]);
  p = __fma_rn(p, f2, kLogPoly[4]);
  p = __fma_rn(p, f2, kLogPoly[5]);
  p = __fma_rn(p, f2, kLogPoly[6]);
  p = __fma_rn(p, f2, kLogPoly[7]);
  p = __dmul_rn(p, f2);
  const double kd = (double)k;
  double res = __fma_rn(kd, 1.90821492927058770002e-10, __dmul_rn(f, p));
  res = __dadd_rn(res, __dmul_rn(2.0, f));
  return __fma_rn(kd, 6.93147180369123816490e-01, res);
}

// order-preserving map double -> uint64 (ascending)
__device__ __forceinline__ unsigned long long ord_f64(double x) {
  unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ unsigned int ord_f32(float x) {
  unsigned int b = __float_as_uint(x);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

template <int G>
__device__ __forceinline__ double group_max(double v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int G>
__device__ __forceinline__ double group_min(double v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int G>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// The log-sum of a state is formed as  max + log1p(sum of the OTHER terms), which
// for two terms is exactly Kaldi's LogAdd (max + log1p(exp(-|d|))) and for more
// terms rounds once instead of once per pair.  One lane of the group (the lowest
// whose local maximum is the group maximum) leaves its arg-max term out.
template <int G>
__device__ __forceinline__ bool elect_max_lane(double local_m, double m, int lane) {
  const unsigned int bal = __ballot_sync(0xffffffffu, local_m == m && m > neg_inf());
  const unsigned int gmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << ((lane / G) * G);
  const unsigned int cand = bal & gmask;
  return cand != 0 && lane == __ffs(cand) - 1;
}

// Last k in [lo, hi] with a[k] <= v, for a[] ascending over [lo, hi] (lo when none is).
template <typename T, typename V>
__device__ __forceinline__ int last_le(const T* a, int lo, int hi, V v) {
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (a[mid] <= v) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// Exclusive prefix sum over the NT threads of a CTA, one tile of a longer scan: returns carry + the
// sum of x over the threads before this one, and adds the tile's sum to carry.  Every thread of the
// CTA calls it (it holds three barriers); warp_sum and carry are __shared__, carry set before a
// barrier.  The shuffles add in T, the carry in C.
template <typename T, int NT, typename C = T>
__device__ __forceinline__ C cta_exclusive_scan(T x, T (&warp_sum)[NT / 32], C& carry) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T incl = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_sum[warp] = incl;
  __syncthreads();
  C add = carry;
#pragma unroll 4  // left to itself the compiler takes 16 values per trip in vector loads (+9 registers)
  for (int w = 0; w < warp; ++w) add += warp_sum[w];
  __syncthreads();
  if (threadIdx.x == NT - 1) carry = add + incl;
  __syncthreads();
  return add + incl - x;
}

__device__ __forceinline__ int4 ld_stream(const int4* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

}  // namespace klu
#endif
