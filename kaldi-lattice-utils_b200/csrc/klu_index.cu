// klu_index.cu -- arc-posterior emit, sort-by-key, segmented log-add and output
// ordering for the word-level index tools (SURVEY.md K6, K7, K8):
//
//   KLU_SEGMENT     kwsbin2/lattice-word-index-segment.cc:134-177 (accumulate),
//                   :96-128 (flatten + sort by logp desc, word, t0, t1)
//   KLU_POSITION    kwsbin2/lattice-word-index-position.cc:135-190, :100-129
//   KLU_FRAME_POST  latbin/lattice-to-word-frame-post.cc:94-135
//
// The reference accumulates into std::map-of-maps; here every valid (arc[, frame
// or length]) pair emits one (key, value) entry in arc order, a stable per-lattice
// radix sort groups equal keys (so each group is folded in the reference's
// accumulation order up to the level renumbering), a segmented LogAdd reduces
// them, and a second stable sort on the ordered bits of the log-probability
// produces the reference's output order (ties fall back to key order because the
// reduced entries are already key-sorted).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {


struct IndexArgs {
  BatchView b;
  CostParams cp;
  int tool;
  int filter_mode, filter_n;
  const int32_t* filter;
  const double* alpha;
  const double* beta;
  const double* alpha2;
  const double* total;
  // --beam
  int use_beam;
  const double* vfwd;
  const double* vbwd;
  const double* best;
  double beam;
  // key layout; drop_key = one bit above every valid key (pruned / unreachable)
  int bits_label, bits_time, bits_len, bits_span;
  unsigned long long drop_key;
  // entries
  const int64_t* ent_base;  // [L] first entry slot of each lattice
  int32_t* arc_ent_off;     // [E] lattice-local first entry of each out-order arc
  int32_t* ent_cnt;         // [L] emitted entries
  unsigned long long* key;
  unsigned int* idx;
  double* val;
  unsigned int* aux;
  int l0;                   // first lattice of the chunk being processed
  long long band_base;      // first band cell of the chunk (alpha2 is chunk-local)
};

__device__ __forceinline__ bool label_valid(const IndexArgs& a, int label) {
  if (label == 0) return false;
  if (a.filter_mode == 0) return true;
  int lo = 0, hi = a.filter_n - 1;
  bool found = false;
  while (lo <= hi) {
    const int mid = (lo + hi) >> 1;
    const int v = a.filter[mid];
    if (v == label) {
      found = true;
      break;
    }
    if (v < label) lo = mid + 1;
    else hi = mid - 1;
  }
  return a.filter_mode == 1 ? found : !found;
}

// entries an out-order arc will emit
__device__ __forceinline__ int arc_entry_count(const IndexArgs& a, int e, int T) {
  const int4 r = a.b.out_rec[e];
  if (a.tool == KLU_FRAME_POST) {
    if (r.w == 0) return 0;
    const int fa = max(a.b.time[a.b.out_src[e]], 0), fb = min(a.b.time[r.x], T);
    return fb > fa ? fb - fa : 0;
  }
  if (a.tool == KLU_BEST_PATH2 || a.tool == KLU_POSITION_POST) {
    if (r.w == 0) return 0;
  } else if (!label_valid(a, r.w)) {
    return 0;
  }
  if (a.tool == KLU_SEGMENT || a.tool == KLU_UTTERANCE) return 1;
  const int s = a.b.out_src[e];
  return (int)(a.b.band_off[s + 1] - a.b.band_off[s]);
}

// One CTA per lattice: exclusive scan of per-arc entry counts.
__global__ void __launch_bounds__(256) k_count_scan(IndexArgs a) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = a.l0 + blockIdx.x;
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const int tid = threadIdx.x;
  const int T = a.b.fr_base[l + 1] - a.b.fr_base[l] - 1;  // frames of the utterance
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = e0; tile < e1; tile += 256) {
    const int e = tile + tid;
    const int c = e < e1 ? arc_entry_count(a, e, T) : 0;
    const int pre = cta_exclusive_scan<int, 256>(c, warp_sum, carry_s);
    if (e < e1) a.arc_ent_off[e] = pre;
  }
  if (tid == 0) a.ent_cnt[l] = carry_s;
}

__device__ __forceinline__ bool emit_arc_pruned(const IndexArgs& a, int l, int s, const int4& r) {
  CostParams cp = a.cp;
  cp.float_sum = 0;
  const double cost = rec_cost(r, cp);
  const double fb = __dadd_rn(a.vfwd[s], __dadd_rn(cost, a.vbwd[r.x]));
  return fb > __dadd_rn(a.best[l], a.beam);
}

// grid (lattices, tiles): one thread per out-order arc.
__global__ void __launch_bounds__(256) k_emit(IndexArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = a.l0 + lt.l;
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const int64_t base = a.ent_base[l];
  for (int e = e0 + lt.tile * blockDim.x + threadIdx.x; e < e1; e += lt.tiles * blockDim.x) {
    const int4 r = a.b.out_rec[e];
    const int s = a.b.out_src[e];
    const int off = a.arc_ent_off[e];
    const unsigned int arc_local = (unsigned int)(e - e0);
    if (a.tool == KLU_SEGMENT) {
      if (!label_valid(a, r.w)) continue;
      const bool dead = a.use_beam && emit_arc_pruned(a, l, s, r);
      // fw[s] + arc_lkh + bw[next], kwsbin2/lattice-word-index-segment.cc:160-162
      const double v = __dadd_rn(__dadd_rn(a.alpha[s], -rec_cost(r, a.cp)), a.beta[r.x]);
      // (word, t0, t1 - t0): the same order as (word, t0, t1) in fewer bits (arcs span a few frames)
      const unsigned long long t0 = (unsigned long long)a.b.time[s], sp = (unsigned long long)(a.b.time[r.x] - a.b.time[s]);
      const unsigned long long k = ((((unsigned long long)r.w << a.bits_time) | t0) << a.bits_span) | sp;
      a.key[base + off] = dead ? a.drop_key : k;
      a.val[base + off] = v;
      a.aux[base + off] = arc_local;
      a.idx[base + off] = (unsigned int)off;
    } else if (a.tool == KLU_UTTERANCE) {
      // one entry per valid arc, grouped by word; the per-word score is computed
      // by k_utt_tasks from the sorted arc lists
      if (!label_valid(a, r.w)) continue;
      const bool dead = a.use_beam && emit_arc_pruned(a, l, s, r);
      a.key[base + off] = dead ? a.drop_key : (unsigned long long)r.w;
      a.val[base + off] = 0.0;
      a.aux[base + off] = arc_local;
      a.idx[base + off] = (unsigned int)off;
    } else if (a.tool == KLU_FRAME_POST) {
      if (r.w == 0) continue;
      const int T = a.b.fr_base[l + 1] - a.b.fr_base[l] - 1;
      const int t0 = max(a.b.time[s], 0), t1 = min(a.b.time[r.x], T);
      if (t1 <= t0) continue;
      // fw[u] + bw[next] - (float)(g + a), latbin/lattice-to-word-frame-post.cc:102-104
      const double v = __dadd_rn(__dadd_rn(a.alpha[s], a.beta[r.x]), -rec_cost(r, a.cp));
      for (int k = t0; k < t1; ++k) {
        const int o = off + (k - t0);
        a.key[base + o] = ((unsigned long long)k << a.bits_label) | (unsigned long long)r.w;
        a.val[base + o] = v;
        a.aux[base + o] = arc_local;
        a.idx[base + o] = (unsigned int)o;
      }
    } else {  // KLU_POSITION, KLU_BEST_PATH2, KLU_POSITION_POST: one entry per (arc, #labels before it)
      const bool plain = a.tool == KLU_BEST_PATH2 || a.tool == KLU_POSITION_POST;
      if (plain ? (r.w == 0) : !label_valid(a, r.w)) continue;
      const int w = (int)(a.b.band_off[s + 1] - a.b.band_off[s]);
      if (w <= 0) continue;
      const bool dead = a.use_beam && emit_arc_pruned(a, l, s, r);
      const int lo = a.b.band_lo[s];
      const double tail = __dadd_rn(-rec_cost(r, a.cp), 0.0);
      for (int i = 0; i < w; ++i) {
        const double al = a.alpha2[a.b.band_off[s] - a.band_base + i];
        // fw[(len,s)] + arc_lkh + bw[next] (position tool, :162-163) or
        // fw[u] + bw[v] - cost (best-path2, :134); beta of the unfolded lattice = beta[next]
        // position-post: fw[u] + bw[next] - (float)(g + a), latbin/lattice-to-word-position-post.cc:111-113
        const double v = plain ? __dadd_rn(__dadd_rn(al, a.beta[r.x]), tail)
                               : __dadd_rn(__dadd_rn(al, tail), a.beta[r.x]);
        // position-post groups by position first: key = (state_len[next] = lo + i + 1, word)
        const unsigned long long k = a.tool == KLU_POSITION_POST
                                         ? (((unsigned long long)(lo + i + 1) << a.bits_label) | (unsigned long long)r.w)
                                         : (((unsigned long long)r.w << a.bits_len) | (unsigned long long)(lo + i));
        const int o = off + i;
        a.key[base + o] = (dead || !(al > neg_inf())) ? a.drop_key : k;
        a.val[base + o] = v;
        a.aux[base + o] = arc_local;
        a.idx[base + o] = (unsigned int)o;
      }
    }
  }
}

struct ReduceArgs {
  BatchView b;
  int tool;
  const int64_t* ent_base;
  const int32_t* ent_cnt;
  const unsigned char* where;
  const unsigned long long *key_a, *key_b;
  const unsigned int *idx_a, *idx_b;
  const double* val;
  const unsigned int* aux;
  const double* total;
  unsigned long long* rkey;
  double* rval;
  unsigned int* raux;
  int32_t* rcnt;
  // second-sort inputs
  unsigned long long* key2;
  unsigned int* key32;  // high half of the f64 order key (what the order sort looks at)
  unsigned int* idx2;
  int bits_label;
  unsigned long long drop_key;
  int l0;
  const double* beta;  // best-path2 normalises by bw[start]
  double* val_rw;      // best-path2: per-entry cost written back over the values
  int32_t* tile_heads;  // per 256-entry tile: key-run heads in it, then (k_reduce_offsets) heads before it
};

// slot of tile t of chunk-local lattice ll in tile_heads (entry bases are not tile aligned:
// one spare slot per lattice keeps the ranges apart)
__device__ __forceinline__ int64_t tile_slot(const ReduceArgs& a, int l, int t) {
  return (a.ent_base[l] >> 8) + (l - a.l0) + t;
}

// Fold each run of equal keys with LogAdd (in sorted = emission order), subtract the
// lattice total, compact, and write the sort key of the output ordering.  Tiles of 256
// entries are independent CTAs (grid: tiles x lattices): k_reduce_count counts the run
// heads of every tile, k_reduce_offsets turns the counts of a lattice into output offsets
// (and the lattice's number of unique keys), k_reduce does the folding -- the head of a
// run owns it to its end, also past the end of its tile.
// Streaming log-sum-exp over the values of one key run: a running maximum m and the sum s
// of exp(v - m), rescaled when the maximum moves -- one cheap exp per term where a chain
// of Kaldi LogAdd calls costs an exp and a log1p each.  The callers keep LogAdd itself for
// runs of one or two terms (bit-identical to the reference there); longer runs agree with
// the reference's chain to ~1e-15.
struct RunSum {
  double m, s;
  __device__ RunSum() : m(neg_inf()), s(0.0) {}
  __device__ void add(double v) {
    if (v == neg_inf()) return;
    if (v <= m) {
      s += fast_exp(v - m);
    } else {
      s = (m == neg_inf() ? 0.0 : s * fast_exp(m - v)) + 1.0;
      m = v;
    }
  }
  __device__ double value() const { return m == neg_inf() ? neg_inf() : m + fast_log(s); }
};

__global__ void __launch_bounds__(256) k_reduce_count(ReduceArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = a.l0 + lt.l;
  const int n = a.ent_cnt[l];
  const unsigned long long* key = (a.where[l] ? a.key_b : a.key_a) + a.ent_base[l];
  for (int tile = lt.tile * 256; tile < n; tile += lt.tiles * 256) {
    const int i = tile + threadIdx.x;
    bool head = false;
    if (i < n) {
      const unsigned long long k = key[i];
      head = k != a.drop_key && (i == 0 || key[i - 1] != k);
    }
    const int cnt = __syncthreads_count(head);
    if (threadIdx.x == 0) a.tile_heads[tile_slot(a, l, tile >> 8)] = cnt;
  }
}

// One CTA per lattice: exclusive prefix of its tile counts, in place; rcnt = their sum.
__global__ void __launch_bounds__(256) k_reduce_offsets(ReduceArgs a) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = a.l0 + blockIdx.x;
  const int n = a.ent_cnt[l];
  const int ntiles = (n + 255) >> 8;
  int32_t* cnt = a.tile_heads + tile_slot(a, l, 0);
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int t0 = 0; t0 < ntiles; t0 += 256) {
    const int t = t0 + tid;
    const int v = t < ntiles ? cnt[t] : 0;
    const int pre = cta_exclusive_scan<int, 256>(v, warp_sum, carry_s);
    if (t < ntiles) cnt[t] = pre;
  }
  if (tid == 0) a.rcnt[l] = carry_s;
}

__global__ void __launch_bounds__(256) k_reduce(ReduceArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  __shared__ int warp_sum[8];
  // the tile's keys, values and arc ranks, staged by all threads at once: the run heads
  // below then walk their runs in shared memory instead of a chain of dependent global
  // gathers (key -> index -> value); only the part of a run past the tile reads global
  __shared__ unsigned long long s_key[256];
  __shared__ double s_val[256];
  __shared__ unsigned int s_aux[256];
  const int l = a.l0 + lt.l;
  const int n = a.ent_cnt[l];
  const int64_t base = a.ent_base[l];
  const unsigned long long* key = (a.where[l] ? a.key_b : a.key_a) + base;
  const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + base;
  const double* val = a.val + base;
  const unsigned int* aux = a.aux + base;
  const double total = a.total[l];
  const int e0 = a.b.e_off[l];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int tile = lt.tile * 256; tile < n; tile += lt.tiles * 256) {
    const int i = tile + tid;
    unsigned long long k = a.drop_key;
    bool head = false;
    if (i < n) {
      k = key[i];
      head = k != a.drop_key && (i == 0 || key[i - 1] != k);
      const unsigned int j0 = idx[i];
      s_key[tid] = k;
      s_val[tid] = val[j0];
      s_aux[tid] = aux[j0];
    }
    const int tile_end = min(n, tile + 256);
    auto key_at = [&](int q) { return q < tile_end ? s_key[q - tile] : key[q]; };
    auto val_at = [&](int q) { return q < tile_end ? s_val[q - tile] : val[idx[q]]; };
    auto aux_at = [&](int q) { return q < tile_end ? s_aux[q - tile] : aux[idx[q]]; };
    int x = head ? 1 : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    int add = a.tile_heads[tile_slot(a, l, tile >> 8)];  // heads of this lattice before the tile
    for (int w = 0; w < warp; ++w) add += warp_sum[w];
    if (head && a.tool == KLU_UTTERANCE) {
      // run of arcs carrying word k: record where it starts, how long it is and
      // the span of source levels it covers
      const int slot = add + x - 1;
      int q = i, lo = 0x7fffffff, hi = -1;
      for (; q < n && key[q] == k; ++q) {
        const int lev = a.b.level[a.b.out_src[e0 + aux[idx[q]]]];
        lo = min(lo, lev);
        hi = max(hi, lev);
      }
      a.rkey[base + slot] = k;
      a.rval[base + slot] = 0.0;
      a.raux[base + slot] = (unsigned int)i;
      a.key2[base + slot] = ((unsigned long long)(unsigned int)lo << 32) | (unsigned long long)(unsigned int)hi;
      a.idx2[base + slot] = (unsigned int)(q - i);
    } else if (head && a.tool == KLU_BEST_PATH2) {
      // latbin/lattice-best-path2.cc:122-147,175: posterior of (label, position),
      // clamped to <= 0, turned into the float cost 1 - P of every arc carrying it
      const int slot = add + x - 1;
      double sum = s_val[tid];
      int q = i + 1;
      if (q + 1 < n && key_at(q + 1) == k) {  // three or more terms
        RunSum rs;
        rs.add(sum);
        for (; q < n && key_at(q) == k; ++q) rs.add(val_at(q));
        sum = rs.value();
      } else {
        for (; q < n && key_at(q) == k; ++q) sum = log_add(sum, val_at(q));
      }
      const double post = fmin(0.0, sum - a.beta[a.b.s_off[l]]);
      double ls;  // LogSub(0, post) [ext]
      if (post >= 0.0) ls = neg_inf();
      else {
        ls = log(1.0 - exp(post));
        if (ls != ls) ls = neg_inf();
      }
      const double cost = (double)(float)exp(ls);
      double* vw = a.val_rw + base;
      for (int t = i; t < q; ++t) vw[idx[t]] = cost;
      a.rkey[base + slot] = k;
      a.rval[base + slot] = post;
      a.raux[base + slot] = 0;
    } else if (head) {
      const int slot = add + x - 1;
      double sum = s_val[tid];
      double bestv = sum;
      unsigned int besta = s_aux[tid];
      const bool longrun = i + 2 < n && key_at(i + 2) == k;  // three or more terms
      RunSum rs;
      if (longrun) rs.add(sum);
      for (int q = i + 1; q < n && key_at(q) == k; ++q) {
        const double v = val_at(q);
        if (longrun) rs.add(v);
        else sum = log_add(sum, v);
        if (a.tool == KLU_POSITION) {
          // strict '>' in reference iteration order (input state, arc order):
          // kwsbin2/lattice-word-index-position.cc:178
          const unsigned int ar = aux_at(q);
          if (v > bestv || (v == bestv && a.b.out_orig[e0 + ar] < a.b.out_orig[e0 + besta])) {
            bestv = v;
            besta = ar;
          }
        }
      }
      if (longrun) sum = rs.value();
      double logp = sum - total;
      a.rkey[base + slot] = k;
      a.rval[base + slot] = logp;
      a.raux[base + slot] = besta;
      logp = logp + 0.0;  // -0.0 and +0.0 compare equal in the reference's sort
      if (a.tool == KLU_FRAME_POST || a.tool == KLU_POSITION_POST) {
        const float f = (float)logp + 0.0f;
        a.key2[base + slot] = ((k >> a.bits_label) << 32) | (unsigned long long)(~ord_f32(f));
      } else {
        a.key32[base + slot] = (unsigned int)((~ord_f64(logp)) >> 32);
      }
      a.idx2[base + slot] = (unsigned int)slot;
    }
    __syncthreads();  // the staging arrays are rewritten by the next tile
  }
}

// The order sort looks at the high half of the f64 keys only (32-bit keys: half the radix
// passes, a third less traffic per pass).  Elements whose keys agree there (log-posteriors
// equal to ~1e-6 relative: a handful per lattice) are left in input order by the stable
// sort; here every such run is put in full-key order -- the full key is read back from the
// reduced values -- by a stable insertion sort, one thread per run.
struct OrderFixArgs {
  const int64_t* seg_base;
  const int32_t* seg_cnt;
  const unsigned char* where;
  unsigned int *key_a, *key_b;
  unsigned int *val_a, *val_b;
  const double* rval;
};

__global__ void __launch_bounds__(256) k_order_fixup(OrderFixArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = a.seg_cnt[l];
  const int64_t base = a.seg_base[l];
  const unsigned int* K = (a.where[l] ? a.key_b : a.key_a) + base;
  unsigned int* V = (a.where[l] ? a.val_b : a.val_a) + base;
  const double* rv = a.rval + base;
  for (int i = lt.tile * blockDim.x + threadIdx.x; i + 1 < n; i += lt.tiles * blockDim.x) {
    const unsigned int t = K[i];
    if ((i > 0 && K[i - 1] == t) || K[i + 1] != t) continue;  // not the head of a run
    int j = i + 1;
    while (j < n && K[j] == t) {  // insert element j into the ordered [i, j)
      const unsigned int v = V[j];
      const unsigned long long k = ~ord_f64(rv[v] + 0.0);
      int q = j;
      while (q > i && (~ord_f64(rv[V[q - 1]] + 0.0)) > k) {
        V[q] = V[q - 1];
        --q;
      }
      V[q] = v;
      ++j;
    }
  }
}

struct GatherArgs {
  BatchView b;
  int tool;
  const int64_t* ent_base;
  const int32_t* rcnt;
  const int64_t* res_off;
  const unsigned char* where;
  const unsigned int *idx_a, *idx_b;
  const unsigned long long* rkey;
  const double* rval;
  const unsigned int* raux;
  int bits_label, bits_time, bits_len, bits_span;
  int32_t *c0, *c1, *c2, *c3;
  double* v;
  float* vf;
  int l0;
};

__global__ void __launch_bounds__(256) k_gather(GatherArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = a.l0 + lt.l;
  const int n = a.rcnt[l];
  const int64_t base = a.ent_base[l];
  const int64_t out = a.res_off[l];
  const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + base;
  const int e0 = a.b.e_off[l];
  for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
    const unsigned int j = idx[i];
    const unsigned long long k = a.rkey[base + j];
    const double logp = a.rval[base + j];
    if (a.tool == KLU_UTTERANCE) {
      a.c0[out + i] = (int32_t)k;
      a.v[out + i] = logp;
    } else if (a.tool == KLU_SEGMENT) {
      const unsigned long long tm = (1ULL << a.bits_time) - 1ULL, sm = (1ULL << a.bits_span) - 1ULL;
      const int32_t t0 = (int32_t)((k >> a.bits_span) & tm);
      a.c0[out + i] = (int32_t)(k >> (a.bits_time + a.bits_span));
      a.c1[out + i] = t0;
      a.c2[out + i] = t0 + (int32_t)(k & sm);
      a.v[out + i] = logp;
    } else if (a.tool == KLU_POSITION) {
      const unsigned long long lm = (1ULL << a.bits_len) - 1ULL;
      const int e = e0 + (int)a.raux[base + j];
      a.c0[out + i] = (int32_t)(k >> a.bits_len);
      a.c1[out + i] = (int32_t)(k & lm) + 1;  // 1-based position, :107
      a.c2[out + i] = a.b.time[a.b.out_src[e]];
      a.c3[out + i] = a.b.time[a.b.out_rec[e].x];
      a.v[out + i] = logp;
    } else {  // frame post / position post (0-based position index)
      const unsigned long long lm = (1ULL << a.bits_label) - 1ULL;
      a.c0[out + i] = (int32_t)(k >> a.bits_label) - (a.tool == KLU_POSITION_POST ? 1 : 0);
      a.c1[out + i] = (int32_t)(k & lm);
      a.vf[out + i] = (float)logp;
    }
  }
}

// ---------------------------------------------------------------- utterance ---
// kwsbin2/lattice-word-index-utterance.cc:161-180 composes the lattice with a
// 2-state "seen w" automaton per word and runs a backward pass on the product.
// Equivalent first-occurrence form (SURVEY.md Appendix B.2):
//   P(w occurs) = sum over arcs a labelled w of  A_w[src(a)] * exp(-cost(a)) * beta[dst(a)]
// where A_w is the forward score over paths that use no w arc.  A_w equals alpha up
// to the first level holding a w arc, so only the levels between the first and the
// last w arc are recomputed (into a per-warp scratch strip).
struct UttArgs {
  BatchView b;
  CostParams cp;
  int l0, nl;
  const int64_t* ent_base;
  const int32_t* rcnt;
  const unsigned char* where;
  const unsigned int *idx_a, *idx_b;
  const unsigned int* aux;
  const unsigned long long* rkey;
  const unsigned int* raux;
  double* rval;
  unsigned long long* key2;
  unsigned int* key32;
  unsigned int* idx2;
  const double* alpha;
  const double* beta;
  double* scratch;
  int max_states;
  int use_beam;
  const double* vfwd;
  const double* vbwd;
  const double* best;
  double beam;
  int* counter;
  const int64_t* res_off;  // [L+1] words (output rows) of the lattices before each one
};

__device__ __forceinline__ bool utt_arc_pruned(const UttArgs& a, int l, int src, int dst, const int4& r) {
  CostParams cp = a.cp;
  cp.float_sum = 0;
  const double fb = __dadd_rn(a.vfwd[src], __dadd_rn(rec_cost(r, cp), a.vbwd[dst]));
  return fb > __dadd_rn(a.best[l], a.beam);
}

template <int G>
__global__ void __launch_bounds__(256) k_utt_tasks(UttArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int SPW = 32 / G;
  const int grp = lane / G, sl = lane % G;
  double* anw = a.scratch + ((size_t)blockIdx.x * 8 + warp) * (size_t)a.max_states;
  const BatchView& b = a.b;
  // Work items are (lattice, word) pairs, numbered through the prefix of the lattices' word
  // counts (res_off) and handed out four at a time to the WARPS of the whole grid: a batch of a
  // few deep lattices (tens of thousands of words each) fills the machine like one of many
  // shallow ones does.
  const long long t_begin = a.res_off[a.l0], t_end = a.res_off[a.l0 + a.nl];
  int l = a.l0;
  for (;;) {
    unsigned int chunk = 0;
    if (lane == 0) chunk = atomicAdd(reinterpret_cast<unsigned int*>(a.counter), 4u);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    const long long tc = t_begin + (long long)chunk;
    if (tc >= t_end) break;
    l = last_le(a.res_off, a.l0, a.l0 + a.nl - 1, tc);  // lattice of the chunk's first item
    for (long long t = tc; t < min(tc + 4, t_end); ++t) {
      while (a.res_off[l + 1] <= t) ++l;
      const int slot = (int)(t - a.res_off[l]);
      const int64_t base = a.ent_base[l];
      const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + base;
      const unsigned int* aux = a.aux + base;
      const int e0 = b.e_off[l], s0 = b.s_off[l];
      const int* lv = b.lvl_start + b.lvl_off[l];
      const double total = a.beta[s0];  // bw_lkh[clat->Start()], :123
      const int w = (int)a.rkey[base + slot];
      const int start = (int)a.raux[base + slot];
      const int len = (int)a.idx2[base + slot];
      const unsigned long long span = a.key2[base + slot];
      const int first = (int)(span >> 32), last = (int)(span & 0xffffffffu);
      const int sb = lv[first + 1];  // first state whose no-w forward score may differ from alpha
      for (int j = first + 1; j <= last; ++j) {
        const int a0 = lv[j], a1 = lv[j + 1];
        for (int bs = a0; bs < a1; bs += SPW) {
          const int s = bs + grp;
          const bool act = s < a1;
          const int i0 = act ? b.in_off[s] : 0, i1 = act ? b.in_off[s + 1] : 0;
          double m = neg_inf();
          int arg = -1;
          for (int e = i0 + sl; e < i1; e += G) {
            const int4 r = __ldg(b.in_rec + e);
            if (r.w == w) continue;
            if (a.use_beam && utt_arc_pruned(a, l, r.x, s, r)) continue;
            const double x = (r.x < sb ? a.alpha[r.x] : anw[r.x - sb]) - rec_cost(r, a.cp);
            if (x > m) {
              m = x;
              arg = e;
            }
          }
          const double lm = m;
          m = group_max<G>(m);
          if (!elect_max_lane<G>(lm, m, lane)) arg = -1;
          double sum = 0.0;
          if (m > neg_inf()) {
            for (int e = i0 + sl; e < i1; e += G) {
              if (e == arg) continue;
              const int4 r = __ldg(b.in_rec + e);
              if (r.w == w) continue;
              if (a.use_beam && utt_arc_pruned(a, l, r.x, s, r)) continue;
              sum += exp((r.x < sb ? a.alpha[r.x] : anw[r.x - sb]) - rec_cost(r, a.cp) - m);
            }
          }
          sum = group_sum<G>(sum);
          if (act && sl == 0) anw[s - sb] = (m > neg_inf()) ? m + log1p(sum) : neg_inf();
        }
        __syncwarp();
      }
      double acc = neg_inf();
      for (int q = lane; q < len; q += 32) {
        const int e = e0 + (int)aux[idx[start + q]];
        const int4 r = b.out_rec[e];
        const int src = b.out_src[e];
        const double fw = src < sb ? a.alpha[src] : anw[src - sb];
        acc = log_add(acc, __dadd_rn(__dadd_rn(fw, -rec_cost(r, a.cp)), a.beta[r.x]));
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc = log_add(acc, __shfl_xor_sync(0xffffffffu, acc, o));
      __syncwarp();
      if (lane == 0) {
        const double logp = acc - total;
        a.rval[base + slot] = logp;
        a.key32[base + slot] = (unsigned int)((~ord_f64(logp + 0.0)) >> 32);
        a.idx2[base + slot] = (unsigned int)slot;
      }
      __syncwarp();
    }
  }
}

int bits_for(int64_t maxv) {
  int b = 1;
  while (b < 63 && ((int64_t)1 << b) <= maxv) ++b;
  return b;
}

}  // namespace

int run_index_tool(klu_ctx* c, int tool, const klu_opts* o) {
  const int32_t L = c->L;
  const bool needs_times = tool != KLU_FWD_BWD && tool != KLU_UTTERANCE && tool != KLU_POSITION_POST;  // best-path2 reports frames (:102)
  if (needs_times)
    for (int32_t l = 0; l < L; ++l)
      if (!c->h_times_ok[l]) {
        // CompactLatticeStateTimes [ext] KALDI_ASSERTs on this
        set_error("lattice " + std::to_string(l) + ": inconsistent state times (lattice is not aligned)");
        return 1;
      }
  const bool use_beam = tool != KLU_FRAME_POST && tool != KLU_FWD_BWD && tool != KLU_BEST_PATH2 &&
                        tool != KLU_POSITION_POST && o->beam != INFINITY;
  if (use_beam && !(o->beam > 0.0f)) {
    set_error("--beam must be positive");  // KALDI_ASSERT(beam > 0.0) in PruneLattice [ext]
    return 1;
  }
  CostParams cp = make_cost_params(o, false);
  if (use_beam) KLU_TRY(run_tropical_sweeps(c, cp));
  // the utterance tool scores with ComputeCompactLatticeBetas [ext]: float-summed costs
  if (tool == KLU_UTTERANCE) cp.float_sum = 1;
  KLU_TRY(run_log_sweeps(c, cp, use_beam, o->beam));
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = 0;
  if (tool == KLU_FWD_BWD || L == 0) return 0;

  // ---- chunk plan: contiguous lattice ranges with bounded scratch ----
  // Entries per chunk (~92 B of scratch each).  The kernels downstream work one CTA or warp per
  // lattice, so a chunk should hold as many lattices as memory allows: half of what is free
  // (counting the scratch this context already holds), between 2^28 and 2^30 entries.
  int64_t kEntryBudget = (int64_t)1 << 28;
  {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      size_t held = 0;
      for (const DevBuf& b : c->d_scratch) held += b.cap;
      const int64_t fit = (int64_t)((free_b + held) / 2 / 92);
      kEntryBudget = std::min<int64_t>((int64_t)1 << 30, std::max<int64_t>(kEntryBudget, fit));
    }
  }
  if (const char* env = getenv("KLU_ENTRY_BUDGET")) kEntryBudget = std::max<long long>(1, atoll(env));  // tests
  const int64_t kBandBudget = (int64_t)1 << 30;   // (state,len) cells per chunk (8 B each)
  std::vector<int64_t> ent_base(L + 1, 0);        // chunk-local first entry slot of each lattice
  std::vector<int32_t> chunk_first;
  {
    int64_t acc = 0, band_acc = 0;
    chunk_first.push_back(0);
    for (int32_t l = 0; l < L; ++l) {
      const int64_t cap = (tool == KLU_SEGMENT || tool == KLU_UTTERANCE) ? (c->h_e_off[l + 1] - c->h_e_off[l])
                          : tool == KLU_FRAME_POST ? c->h_cap_frame[l] : c->h_cap_pos[l];
      const int64_t band = (tool == KLU_POSITION || tool == KLU_BEST_PATH2 || tool == KLU_POSITION_POST)
                               ? c->h_band_off[l + 1] - c->h_band_off[l] : 0;
      if (cap >= ((int64_t)1 << 31)) {
        set_error("lattice " + std::to_string(l) + ": more than 2^31 index entries");
        return 1;
      }
      if (l > chunk_first.back() && (acc + cap > kEntryBudget || band_acc + band > kBandBudget)) {
        chunk_first.push_back(l);
        acc = 0;
        band_acc = 0;
      }
      ent_base[l] = acc;
      acc += cap;
      band_acc += band;
    }
    chunk_first.push_back(L);
  }
  int64_t N = 1;  // largest chunk
  for (size_t k = 0; k + 1 < chunk_first.size(); ++k) {
    const int32_t last = chunk_first[k + 1] - 1;
    const int64_t cap = (tool == KLU_SEGMENT || tool == KLU_UTTERANCE) ? (c->h_e_off[last + 1] - c->h_e_off[last])
                        : tool == KLU_FRAME_POST ? c->h_cap_frame[last] : c->h_cap_pos[last];
    N = std::max(N, ent_base[last] + cap);
  }
  const bool single_chunk = chunk_first.size() == 2;
  enum { S_BASE = 0, S_ARCOFF, S_CNT, S_KEYA, S_KEYB, S_IDXA, S_IDXB, S_VAL, S_AUX, S_WHERE, S_RCNT, S_R };
  KLU_TRY(c->d_scratch[S_BASE].reserve(sizeof(int64_t) * (L + 1)));
  KLU_TRY(c->d_scratch[S_ARCOFF].reserve(sizeof(int32_t) * std::max<int64_t>(c->E, 1)));
  KLU_TRY(c->d_scratch[S_CNT].reserve(sizeof(int32_t) * L));
  KLU_TRY(c->d_scratch[S_KEYA].reserve(sizeof(int64_t) * N));
  KLU_TRY(c->d_scratch[S_KEYB].reserve(sizeof(int64_t) * N));
  KLU_TRY(c->d_scratch[S_IDXA].reserve(sizeof(int32_t) * N));
  KLU_TRY(c->d_scratch[S_IDXB].reserve(sizeof(int32_t) * N));
  KLU_TRY(c->d_scratch[S_VAL].reserve(sizeof(double) * N));
  KLU_TRY(c->d_scratch[S_AUX].reserve(sizeof(int32_t) * N));
  KLU_TRY(c->d_scratch[S_WHERE].reserve(2 * (size_t)L));
  KLU_TRY(c->d_scratch[S_RCNT].reserve(sizeof(int32_t) * L));
  // reduced entries: key (8) + val (8) + aux (4) per slot
  KLU_TRY(c->d_scratch[S_R].reserve(20 * (size_t)N + 64));
  KLU_TRY(c->d_res[6].reserve(12 * (size_t)N));  // ordering-sort keys: 64-bit (float tools) | 32-bit (f64 tools)
  KLU_TRY(c->d_res[7].reserve(sizeof(int32_t) * N));  // ordering-sort values
  KLU_TRY(c->d_res[5].reserve(sizeof(int64_t) * (L + 1)));
  KLU_CUDA(cudaMemcpyAsync(c->d_scratch[S_BASE].p, ent_base.data(), sizeof(int64_t) * (L + 1),
                           cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemsetAsync(c->d_res[5].p, 0, sizeof(int64_t), c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // ent_base is a stack object

  int fmode = 0, fn = 0;
  if (tool != KLU_FRAME_POST && tool != KLU_BEST_PATH2 && tool != KLU_POSITION_POST)
    KLU_TRY(upload_filter(c, o, &fmode, &fn));

  IndexArgs a;
  a.b = c->view();
  a.cp = make_cost_params(o, tool == KLU_FRAME_POST || tool == KLU_POSITION_POST);  // these add g + a in float
  a.tool = tool;
  a.filter_mode = fmode;
  a.filter_n = fn;
  a.filter = c->d_filter.as<int32_t>();
  a.alpha = c->d_alpha.as<double>();
  a.beta = c->d_beta.as<double>();
  a.total = c->d_total.as<double>();
  a.use_beam = use_beam ? 1 : 0;
  a.vfwd = c->d_vfwd.as<double>();
  a.vbwd = c->d_vbwd.as<double>();
  a.best = c->d_best.as<double>();
  a.beam = (double)o->beam;
  a.bits_label = bits_for(c->max_label);
  a.bits_time = bits_for(c->max_time);
  a.bits_len = bits_for(c->max_len);
  a.bits_span = bits_for(c->max_span);
  a.ent_base = c->d_scratch[S_BASE].as<int64_t>();
  a.arc_ent_off = c->d_scratch[S_ARCOFF].as<int32_t>();
  a.ent_cnt = c->d_scratch[S_CNT].as<int32_t>();
  a.key = c->d_scratch[S_KEYA].as<unsigned long long>();
  a.idx = c->d_scratch[S_IDXA].as<unsigned int>();
  a.val = c->d_scratch[S_VAL].as<double>();
  a.aux = c->d_scratch[S_AUX].as<unsigned int>();
  int key_bits = 0;
  if (tool == KLU_UTTERANCE) key_bits = a.bits_label;
  else if (tool == KLU_SEGMENT) key_bits = a.bits_label + a.bits_time + a.bits_span;
  else if (tool == KLU_POSITION || tool == KLU_BEST_PATH2 || tool == KLU_POSITION_POST)
    key_bits = a.bits_label + a.bits_len + (tool == KLU_POSITION_POST ? 1 : 0);  // positions run to max_len inclusive
  else key_bits = a.bits_time + a.bits_label;
  if (key_bits > 62 || (tool == KLU_FRAME_POST && a.bits_time > 31) || (tool == KLU_POSITION_POST && a.bits_len > 30)) {
    set_error("index key does not fit 62 bits (labels/times too large)");
    return 1;
  }
  a.drop_key = 1ULL << key_bits;

  int64_t res_cap = 0, res_used = 0;  // result columns: capacity / entries known to be in use
  auto grow_results = [&](int64_t need) -> int {
    if (need <= res_cap) return 0;
    const int64_t want = std::max<int64_t>(need, res_cap * 2);
    for (int i = 0; i < 5; ++i) {
      const size_t w = i == 4 ? 8 : 4;
      if (c->d_res[i].cap >= (size_t)want * w) continue;
      DevBuf nb;
      KLU_TRY(nb.reserve((size_t)want * w));
      if (res_used > 0)
        KLU_CUDA(cudaMemcpyAsync(nb.p, c->d_res[i].p, (size_t)res_used * w, cudaMemcpyDeviceToDevice, c->stream));
      KLU_CUDA(cudaStreamSynchronize(c->stream));
      c->d_res[i].release();
      c->d_res[i] = nb;
    }
    res_cap = want;
    return 0;
  };

  for (size_t k = 0; k + 1 < chunk_first.size(); ++k) {
    const int32_t l0 = chunk_first[k], l1 = chunk_first[k + 1];
    const int nl = l1 - l0;
    if (nl <= 0) continue;
    a.l0 = l0;
    a.band_base = 0;
    if (tool == KLU_POSITION || tool == KLU_BEST_PATH2 || tool == KLU_POSITION_POST) {
      KLU_TRY(run_banded_alpha(c, cp, use_beam, o->beam, l0, l1));
      a.band_base = c->h_band_off[l0];
    }
    a.alpha2 = c->d_alpha2.as<double>();
    {
      KLU_LAUNCH(c, "k_count_scan");
      k_count_scan<<<nl, 256, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_count_scan"));
    int64_t max_arcs = 0, chunk_cap = 0;
    for (int32_t l = l0; l < l1; ++l) max_arcs = std::max(max_arcs, c->h_e_off[l + 1] - c->h_e_off[l]);
    {
      const int32_t last = l1 - 1;
      const int64_t cap = (tool == KLU_SEGMENT || tool == KLU_UTTERANCE)
                              ? (c->h_e_off[last + 1] - c->h_e_off[last])
                              : tool == KLU_FRAME_POST ? c->h_cap_frame[last] : c->h_cap_pos[last];
      chunk_cap = ent_base[last] + cap;
    }
    const int tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
    {
      KLU_LAUNCH(c, "k_emit");
      k_emit<<<dim3(nl, tiles), 256, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_emit"));

    SegSortArgs s1;
    s1.seg_base = a.ent_base + l0;
    s1.seg_cnt = a.ent_cnt + l0;
    s1.key_a = c->d_scratch[S_KEYA].as<unsigned long long>();
    s1.val_a = c->d_scratch[S_IDXA].as<unsigned int>();
    s1.key_b = c->d_scratch[S_KEYB].as<unsigned long long>();
    s1.val_b = c->d_scratch[S_IDXB].as<unsigned int>();
    s1.where = c->d_scratch[S_WHERE].as<unsigned char>() + l0;
    s1.lo_bit = 0;
    s1.hi_bit = key_bits + 1;  // + the drop bit; degenerate digits are skipped per lattice
    {
      KLU_LAUNCH(c, "k_seg_radix_sort");
      KLU_TRY(seg_sort_launch(c, s1, nl, N));
    }
    KLU_TRY(check_launch("k_seg_radix_sort(keys)"));

    ReduceArgs r;
    r.b = a.b;
    r.tool = tool;
    r.l0 = l0;
    r.ent_base = a.ent_base;
    r.ent_cnt = a.ent_cnt;
    r.where = c->d_scratch[S_WHERE].as<unsigned char>();
    r.key_a = s1.key_a;
    r.key_b = s1.key_b;
    r.idx_a = s1.val_a;
    r.idx_b = s1.val_b;
    r.val = a.val;
    r.aux = a.aux;
    r.total = a.total;
    char* rp = c->d_scratch[S_R].as<char>();
    r.rkey = reinterpret_cast<unsigned long long*>(rp);
    r.rval = reinterpret_cast<double*>(rp + 8 * (size_t)N);
    r.raux = reinterpret_cast<unsigned int*>(rp + 16 * (size_t)N);
    r.rcnt = c->d_scratch[S_RCNT].as<int32_t>();
    // the ordering sort's input pair is separate from the first sort's buffers
    // (the reduce reads those); its ping-pong partner is the then-free A side.
    r.key2 = c->d_res[6].as<unsigned long long>();
    r.key32 = reinterpret_cast<unsigned int*>(r.key2 + N);
    r.idx2 = c->d_res[7].as<unsigned int>();
    r.bits_label = a.bits_label;
    r.drop_key = a.drop_key;
    r.beta = a.beta;
    r.val_rw = a.val;
    {
      int64_t max_cap = 1;
      for (int32_t l = l0; l < l1; ++l) max_cap = std::max<int64_t>(max_cap, ent_base[l + 1 < l1 ? l + 1 : l] - ent_base[l]);
      max_cap = std::max<int64_t>(max_cap, chunk_cap - ent_base[l1 - 1]);
      const int rtiles = (int)std::min<int64_t>((max_cap + 255) / 256, 8192);
      KLU_TRY(c->d_tile_heads.reserve(4 * (size_t)((chunk_cap >> 8) + nl + 2)));
      r.tile_heads = c->d_tile_heads.as<int32_t>();
      {
        KLU_LAUNCH(c, "k_reduce_count");
        k_reduce_count<<<dim3(nl, rtiles), 256, 0, c->stream>>>(r);
      }
      KLU_TRY(check_launch("k_reduce_count"));
      {
        KLU_LAUNCH(c, "k_reduce_offsets");
        k_reduce_offsets<<<nl, 256, 0, c->stream>>>(r);
      }
      KLU_TRY(check_launch("k_reduce_offsets"));
      KLU_LAUNCH(c, "k_reduce");
      k_reduce<<<dim3(nl, rtiles), 256, 0, c->stream>>>(r);
    }
    KLU_TRY(check_launch("k_reduce"));
    if (tool == KLU_UTTERANCE) {
      UttArgs u;
      u.b = a.b;
      u.cp = cp;
      u.l0 = l0;
      u.nl = nl;
      u.ent_base = a.ent_base;
      u.rcnt = r.rcnt;
      u.where = r.where;
      u.idx_a = s1.val_a;
      u.idx_b = s1.val_b;
      u.aux = a.aux;
      u.rkey = r.rkey;
      u.raux = r.raux;
      u.rval = r.rval;
      u.key2 = r.key2;
      u.key32 = r.key32;
      u.idx2 = r.idx2;
      u.alpha = a.alpha;
      u.beta = a.beta;
      u.max_states = std::max(1, c->max_states);
      u.use_beam = a.use_beam;
      u.vfwd = a.vfwd;
      u.vbwd = a.vbwd;
      u.best = a.best;
      u.beam = a.beam;
      KLU_TRY(scan_counts(c, r.rcnt, l0, l1, c->d_res[5].as<int64_t>(), "k_scan_counts"));
      u.res_off = c->d_res[5].as<int64_t>();
      const int grid = std::max(1, c->num_sms * 4);
      KLU_TRY(c->d_alpha2.reserve(sizeof(double) * (size_t)grid * 8 * (size_t)u.max_states));
      u.scratch = c->d_alpha2.as<double>();
      KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));
      u.counter = c->d_counter.as<int>();
      const int G = pick_group(c->avg_deg);
      {
        KLU_LAUNCH(c, "k_utt_tasks");
        KLU_DISPATCH_G(G, k_utt_tasks<kG><<<grid, 256, 0, c->stream>>>(u));
      }
      KLU_TRY(check_launch("k_utt_tasks"));
    }
    // f64 order keys (segment, utterance): 32-bit sort on the high half, near-ties settled afterwards;
    // float tools (generic frame-post / position-post): (frame or position, float) in 64 bits
    const bool half_keys = !(tool == KLU_FRAME_POST || tool == KLU_POSITION_POST);
    unsigned char* where2 = c->d_scratch[S_WHERE].as<unsigned char>() + L + l0;
    unsigned int* ord_a = r.idx2;
    unsigned int* ord_b = c->d_scratch[S_IDXA].as<unsigned int>();
    if (half_keys) {
      SegSortArgs32 s2;
      s2.seg_base = a.ent_base + l0;
      s2.seg_cnt = r.rcnt + l0;
      s2.key_a = r.key32;
      s2.val_a = ord_a;
      s2.key_b = c->d_scratch[S_KEYA].as<unsigned int>();
      s2.val_b = ord_b;
      s2.where = where2;
      s2.lo_bit = 0;
      s2.hi_bit = 32;
      {
        KLU_LAUNCH(c, "k_seg_radix_sort");
        KLU_TRY(seg_sort_launch(c, s2, nl, N));
      }
      KLU_TRY(check_launch("k_seg_radix_sort(order)"));
      OrderFixArgs f;
      f.seg_base = s2.seg_base;
      f.seg_cnt = s2.seg_cnt;
      f.where = s2.where;
      f.key_a = s2.key_a, f.key_b = s2.key_b;
      f.val_a = s2.val_a, f.val_b = s2.val_b;
      f.rval = r.rval + 0;
      {
        KLU_LAUNCH(c, "k_order_fixup");
        k_order_fixup<<<dim3(nl, tiles), 256, 0, c->stream>>>(f);
      }
      KLU_TRY(check_launch("k_order_fixup"));
    } else {
      SegSortArgs s2;
      s2.seg_base = a.ent_base + l0;
      s2.seg_cnt = r.rcnt + l0;
      s2.key_a = r.key2;
      s2.val_a = ord_a;
      s2.key_b = c->d_scratch[S_KEYA].as<unsigned long long>();
      s2.val_b = ord_b;
      s2.where = where2;
      s2.lo_bit = 0;
      s2.hi_bit = 64;
      {
        KLU_LAUNCH(c, "k_seg_radix_sort");
        KLU_TRY(seg_sort_launch(c, s2, nl, N));
      }
      KLU_TRY(check_launch("k_seg_radix_sort(order)"));
    }
    KLU_TRY(scan_counts(c, r.rcnt, l0, l1, c->d_res[5].as<int64_t>(), "k_scan_counts"));
    if (single_chunk) {
      KLU_TRY(grow_results(chunk_cap));
    } else {
      int64_t upto = 0;
      KLU_CUDA(cudaMemcpyAsync(&upto, c->d_res[5].as<int64_t>() + l1, sizeof(int64_t), cudaMemcpyDeviceToHost,
                               c->stream));
      KLU_CUDA(cudaStreamSynchronize(c->stream));
      KLU_TRY(grow_results(upto));
      res_used = upto;
    }
    GatherArgs g;
    g.b = a.b;
    g.tool = tool;
    g.l0 = l0;
    g.ent_base = a.ent_base;
    g.rcnt = r.rcnt;
    g.res_off = c->d_res[5].as<int64_t>();
    g.where = c->d_scratch[S_WHERE].as<unsigned char>() + L;
    g.idx_a = ord_a;
    g.idx_b = ord_b;
    g.rkey = r.rkey;
    g.rval = r.rval;
    g.raux = r.raux;
    g.bits_label = a.bits_label;
    g.bits_time = a.bits_time;
    g.bits_len = a.bits_len;
    g.bits_span = a.bits_span;
    g.c0 = c->d_res[0].as<int32_t>();
    g.c1 = c->d_res[1].as<int32_t>();
    g.c2 = c->d_res[2].as<int32_t>();
    g.c3 = c->d_res[3].as<int32_t>();
    g.v = c->d_res[4].as<double>();
    g.vf = c->d_res[4].as<float>();
    {
      KLU_LAUNCH(c, "k_gather");
      k_gather<<<dim3(nl, tiles), 256, 0, c->stream>>>(g);
    }
    KLU_TRY(check_launch("k_gather"));
  }
  c->last_entries = -1;  // known after klu_result_offsets()
  return 0;
}

}  // namespace klu

using namespace klu;

static __global__ void k_unpermute(const double* alpha, const double* beta, const int32_t* old2new, double* oa,
                                   double* ob, int64_t S) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < S; s += stride) {
    const int n = old2new[s];
    oa[s] = alpha[n];
    ob[s] = beta[n];
  }
}

// Lazily brings the per-lattice result offsets of the last run to the host.
static int ensure_offsets(klu_ctx* c) {
  if (c->last_tool < 0) {
    set_error("no results: klu_run has not succeeded on this batch");
    return 1;
  }
  KLU_CUDA(cudaSetDevice(c->device));
  if (c->last_entries >= 0) {
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  }
  c->h_res_off.resize(c->L + 1);
  KLU_CUDA(cudaMemcpyAsync(c->h_res_off.data(), c->d_res[5].p, sizeof(int64_t) * (c->L + 1), cudaMemcpyDeviceToHost,
                           c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  c->last_entries = c->h_res_off[c->L];
  return 0;
}

static int d2h(klu_ctx* c, void* dst, const void* src, size_t bytes) {
  if (!dst || !bytes) return 0;
  KLU_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
  return 0;
}

extern "C" {

int klu_result_offsets(klu_ctx* c, int64_t* entry_off) {
  KLU_TRY(ensure_offsets(c));
  memcpy(entry_off, c->h_res_off.data(), sizeof(int64_t) * (c->L + 1));
  return 0;
}

int klu_fetch_segment(klu_ctx* c, int32_t* word, int32_t* t0, int32_t* t1, double* logp) {
  if (c->last_tool != KLU_SEGMENT) {
    set_error("klu_fetch_segment: last run was not KLU_SEGMENT");
    return 1;
  }
  KLU_TRY(ensure_offsets(c));
  const size_t n = (size_t)c->last_entries;
  KLU_TRY(d2h(c, word, c->d_res[0].p, n * 4));
  KLU_TRY(d2h(c, t0, c->d_res[1].p, n * 4));
  KLU_TRY(d2h(c, t1, c->d_res[2].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 8));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_fetch_position(klu_ctx* c, int32_t* word, int32_t* pos, int32_t* t0, int32_t* t1, double* logp) {
  if (c->last_tool != KLU_POSITION) {
    set_error("klu_fetch_position: last run was not KLU_POSITION");
    return 1;
  }
  KLU_TRY(ensure_offsets(c));
  const size_t n = (size_t)c->last_entries;
  KLU_TRY(d2h(c, word, c->d_res[0].p, n * 4));
  KLU_TRY(d2h(c, pos, c->d_res[1].p, n * 4));
  KLU_TRY(d2h(c, t0, c->d_res[2].p, n * 4));
  KLU_TRY(d2h(c, t1, c->d_res[3].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 8));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_fetch_utterance(klu_ctx* c, int32_t* word, double* logp) {
  if (c->last_tool != KLU_UTTERANCE) {
    set_error("klu_fetch_utterance: last run was not KLU_UTTERANCE");
    return 1;
  }
  KLU_TRY(ensure_offsets(c));
  const size_t n = (size_t)c->last_entries;
  KLU_TRY(d2h(c, word, c->d_res[0].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 8));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_fetch_frame_post(klu_ctx* c, int32_t* num_frames, int32_t* frame, int32_t* word, float* logp) {
  if (c->last_tool != KLU_FRAME_POST) {
    set_error("klu_fetch_frame_post: last run was not KLU_FRAME_POST");
    return 1;
  }
  klu_trace(c, "fetch: waiting for the run");
  KLU_TRY(ensure_offsets(c));
  klu_trace(c, "fetch: download begins");
  const size_t n = (size_t)c->last_entries;
  if (num_frames) memcpy(num_frames, c->h_num_frames.data(), sizeof(int32_t) * c->L);
  // the frame column of the frame-synchronous path is static per batch (klu_frame.cu);
  // the generic pipeline (KLU_GENERIC_FRAME_POST) writes its own
  KLU_TRY(d2h(c, frame, c->frame_col_static ? c->d_fr_gframe.p : c->d_res[0].p, n * 4));
  KLU_TRY(d2h(c, word, c->d_res[1].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 4));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  klu_trace(c, "fetch: done");
  return 0;
}

int klu_fetch_frame_post_csr(klu_ctx* c, int32_t* num_frames, int64_t* frame_row_off, int32_t* word, float* logp) {
  if (c->last_tool != KLU_FRAME_POST) {
    set_error("klu_fetch_frame_post_csr: last run was not KLU_FRAME_POST");
    return 1;
  }
  KLU_TRY(ensure_offsets(c));
  const size_t n = (size_t)c->last_entries;
  const int32_t L = c->L;
  if (num_frames) memcpy(num_frames, c->h_num_frames.data(), sizeof(int32_t) * L);
  if (frame_row_off && c->frame_col_static) {
    // the frame-synchronous path keeps the per-frame row offsets of the batch on the device (klu_frame.cu)
    KLU_TRY(d2h(c, frame_row_off, c->d_fr_gloc.p, 8 * (size_t)c->h_fr_base[L]));
  } else if (frame_row_off) {
    // generic pipeline (KLU_GENERIC_FRAME_POST): count the rows of every frame from its frame column
    std::vector<int32_t> fr(n);
    KLU_TRY(d2h(c, fr.data(), c->d_res[0].p, n * 4));
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    size_t o = 0;
    for (int32_t l = 0; l < L; ++l) {
      const size_t a = (size_t)c->h_res_off[l], e = (size_t)c->h_res_off[l + 1];
      size_t i = a;
      for (int32_t k = 0; k < c->h_num_frames[l]; ++k) {
        frame_row_off[o++] = (int64_t)(i - a);
        while (i < e && fr[i] == k) ++i;
      }
      frame_row_off[o++] = (int64_t)(e - a);
    }
  }
  KLU_TRY(d2h(c, word, c->d_res[1].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 4));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_fetch_length_dist(klu_ctx* c, int32_t* length, float* logp) {
  if (c->last_tool != KLU_LENGTH_DIST) {
    set_error("klu_fetch_length_dist: last run was not KLU_LENGTH_DIST");
    return 1;
  }
  KLU_TRY(ensure_offsets(c));
  const size_t n = (size_t)c->last_entries;
  KLU_TRY(d2h(c, length, c->d_res[0].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 4));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_fetch_position_post(klu_ctx* c, int32_t* num_positions, int32_t* position, int32_t* word, float* logp) {
  if (c->last_tool != KLU_POSITION_POST) {
    set_error("klu_fetch_position_post: last run was not KLU_POSITION_POST");
    return 1;
  }
  KLU_TRY(ensure_offsets(c));
  const size_t n = (size_t)c->last_entries;
  if (num_positions) memcpy(num_positions, c->h_maxlen.data(), sizeof(int32_t) * c->L);
  KLU_TRY(d2h(c, position, c->d_res[0].p, n * 4));
  KLU_TRY(d2h(c, word, c->d_res[1].p, n * 4));
  KLU_TRY(d2h(c, logp, c->d_res[4].p, n * 4));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int klu_fetch_fwd_bwd(klu_ctx* c, double* alpha, double* beta, double* total) {
  if (c->last_tool < 0) {
    set_error("klu_fetch_fwd_bwd: no run");
    return 1;
  }
  KLU_CUDA(cudaSetDevice(c->device));
  // back to the caller's state numbering on the device, then one copy each
  const size_t S = (size_t)c->S;
  if (S) {
    KLU_TRY(c->d_res[6].reserve(16 * S));
    double* tmp = c->d_res[6].as<double>();
    k_unpermute<<<c->num_sms * 4, 256, 0, c->stream>>>(c->d_alpha.as<double>(), c->d_beta.as<double>(),
                                                      c->d_old2new.as<int32_t>(), tmp, tmp + S, (int64_t)S);
    KLU_TRY(check_launch("k_unpermute"));
    if (alpha) KLU_CUDA(cudaMemcpyAsync(alpha, tmp, 8 * S, cudaMemcpyDeviceToHost, c->stream));
    if (beta) KLU_CUDA(cudaMemcpyAsync(beta, tmp + S, 8 * S, cudaMemcpyDeviceToHost, c->stream));
  }
  if (total && c->L)
    KLU_CUDA(cudaMemcpyAsync(total, c->d_total.p, sizeof(double) * c->L, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

}  // extern "C"
