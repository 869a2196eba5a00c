// klu_position.cu -- the (word, position) tools: lattice-word-index-position,
// lattice-to-word-position-post and the posterior stage of lattice-best-path2.
//
//   KLU_POSITION       kwsbin2/lattice-word-index-position.cc:135-190 (accumulate), :100-129 (order)
//   KLU_POSITION_POST  latbin/lattice-to-word-position-post.cc:94-141
//   KLU_BEST_PATH2     latbin/lattice-best-path2.cc:122-147 (posteriors), then klu_bestpath.cu
//
// The reference unfolds the lattice by label count (DisambiguateStateInputSequenceLength,
// fstext/fstext-utils2.h:109-215), runs forward-backward on the unfolded copy and
// accumulates every arc into a std::map keyed by (word, position).  Unfolded, a c2 lattice
// (50 k arcs) has ~10 M arcs; emitting, sorting and reducing one entry per unfolded arc is
// what the first version of this file's tools did.  Here nothing is unfolded and nothing is
// sorted by (word, position):
//   1. the lattice's arcs are grouped by word once (stable segmented radix sort of E keys);
//   2. a word's group covers the positions [min band_lo(src), max band_hi(src)) of its arcs:
//      that range is a row of CELLS, one per (word, position), laid out back to back;
//   3. one thread per cell walks the group's arcs and adds up
//      alpha2[src][position] - cost + beta[dst] over the arcs whose source band holds the
//      position -- consecutive threads are consecutive positions, so the banded alpha is read
//      in contiguous runs and the per-arc record is a broadcast;
//   4. cells that exist (some arc reaches them) are compacted and ordered by log-posterior.
// The cell sums are the reference's map entries; their order of accumulation differs (arcs of a
// word in packed-state order instead of unfolded-state order), which moves a 3+-term sum by
// ~1e-16 relative; one- and two-term sums are Kaldi's LogAdd exactly.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

struct __align__(16) ArcRec {
  long long base;  // alpha2 (chunk-local) index of (source, position) = base + position
  double tail;     // -cost of the arc
  double beta;     // beta[destination]
  int lo, hi;      // positions the source's band holds: [lo, hi)
};

// One (word, position) cell as the ordering / gather stages read it: one 32-byte sector.
struct __align__(16) CellRec {
  double val;               // log-posterior
  unsigned long long key;   // (word, position) packed; position-post: (position + 1, word)
  int t0, t1;               // position index: segment of the best single arc
  unsigned int exists;      // some arc reaches the cell
  unsigned int pad;
};

struct PosArgs {
  BatchView b;
  CostParams cp;
  int tool;
  int filter_mode, filter_n;
  const int32_t* filter;
  const double* beta;
  const double* alpha2;
  const double* total;
  int use_beam;
  const double* vfwd;
  const double* vbwd;
  const double* best;
  double beam;
  int bits_label, bits_len;
  unsigned long long drop_key;
  // ---- whole batch: arcs grouped by word (segments = lattices, indexed by global arc position)
  const int64_t* seg_base;  // [L] first arc of each lattice (64-bit copy of e_off)
  const int32_t* seg_cnt;   // [L]
  unsigned long long *key_a, *key_b;
  unsigned int *idx_a, *idx_b;
  const unsigned char* where;
  int32_t* tile_heads;  // per 256-arc tile: group heads in it, then (prefix) heads before it
  int32_t* ngroups;     // [L]
  // groups of lattice l live at e_off[l] + slot
  int32_t *g_word, *g_start, *g_len, *g_plo, *g_phi, *g_celloff;
  int32_t* q_group;     // [E] group slot of every sorted arc
  long long* lat_cells;  // [L] cells of each lattice
  // ---- chunk
  int l0;
  long long band_base;
  const int64_t* cell_base;  // [L] chunk-local first cell of each lattice
  int e_chunk0;              // first arc of the chunk
  ArcRec* rec;               // [chunk arcs] in sorted order
  CellRec* cell;   // position / position-post
  double* ccost;   // best-path2: float cost 1 - P of the cell, as a double
  int32_t* ctile;  // per 256-cell tile: existing cells in it, then (prefix) existing cells before it
  int32_t* tile_group;  // per 256-cell tile: group of its first cell (k_pos_tile_groups)
  int32_t* rcnt;   // [L] existing cells = output rows
  unsigned long long* key2;  // order keys: 64-bit (position-post) ...
  unsigned int* key32;       // ... or the high half of the f64 key only (position)
  unsigned int* idx2;
  long long* arc_cellbase;  // [E] best-path2: cell of (arc, position) = arc_cellbase[e] + position
};

__device__ __forceinline__ bool pos_label_valid(const PosArgs& a, int label) {
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

// tile slot of (lattice l, tile t) in an array with one spare slot per lattice (segment bases
// are not tile aligned)
__device__ __forceinline__ int64_t tile_slot(const int64_t* base, int l, int l_first, int t) {
  return (base[l] >> 8) + (l - l_first) + t;
}

// grid (lattices, tiles): sort key of every out-order arc = its word (or the drop key)
__global__ void __launch_bounds__(256) k_pos_keys(PosArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const bool plain = a.tool != KLU_POSITION;
  for (int e = e0 + lt.tile * blockDim.x + threadIdx.x; e < e1; e += lt.tiles * blockDim.x) {
    const int4 r = a.b.out_rec[e];
    const int s = a.b.out_src[e];
    bool valid = plain ? r.w != 0 : pos_label_valid(a, r.w);
    if (valid && a.b.band_off[s + 1] <= a.b.band_off[s]) valid = false;  // unreachable source
    if (valid && a.use_beam) {
      CostParams cp = a.cp;
      cp.float_sum = 0;
      const double fb = __dadd_rn(a.vfwd[s], __dadd_rn(rec_cost(r, cp), a.vbwd[r.x]));
      if (fb > __dadd_rn(a.best[l], a.beam)) valid = false;  // PruneLattice [ext] drops the arc
    }
    a.key_a[e] = valid ? (unsigned long long)(unsigned int)r.w : a.drop_key;
    a.idx_a[e] = (unsigned int)(e - e0);
  }
}

// grid (lattices, tiles): group heads per 256-arc tile of the sorted arcs
__global__ void __launch_bounds__(256) k_pos_head_count(PosArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = a.seg_cnt[l];
  const unsigned long long* key = (a.where[l] ? a.key_b : a.key_a) + a.seg_base[l];
  for (int tile = lt.tile * 256; tile < n; tile += lt.tiles * 256) {
    const int i = tile + threadIdx.x;
    bool head = false;
    if (i < n) {
      const unsigned long long k = key[i];
      head = k != a.drop_key && (i == 0 || key[i - 1] != k);
    }
    const int cnt = __syncthreads_count(head);
    if (threadIdx.x == 0) a.tile_heads[tile_slot(a.seg_base, l, 0, tile >> 8)] = cnt;
  }
}

// One CTA per segment: exclusive prefix of its tile counts, in place; total[seg] = their sum.
__global__ void __launch_bounds__(256) k_tile_prefix(const int64_t* base, const long long* n64, const int32_t* n32,
                                                     int l_first, int32_t* tiles, int32_t* total) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = l_first + blockIdx.x;
  const long long n = n64 ? n64[l] : (long long)n32[l];
  const int ntiles = (int)((n + 255) >> 8);
  int32_t* cnt = tiles + tile_slot(base, l, l_first, 0);
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int t0 = 0; t0 < ntiles; t0 += 256) {
    const int t = t0 + tid;
    const int v = t < ntiles ? cnt[t] : 0;
    const int pre = cta_exclusive_scan<int, 256>(v, warp_sum, carry_s);
    if (t < ntiles) cnt[t] = pre;
  }
  if (tid == 0) total[l] = carry_s;
}

// grid (lattices, tiles): the head of a group walks its arcs: word, extent in the sorted list,
// range of positions [plo, phi) its arcs' source bands cover
__global__ void __launch_bounds__(256) k_pos_groups(PosArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  __shared__ int warp_sum[8];
  const int l = lt.l;
  const int n = a.seg_cnt[l];
  const int e0 = a.b.e_off[l];
  const unsigned long long* key = (a.where[l] ? a.key_b : a.key_a) + a.seg_base[l];
  const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + a.seg_base[l];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int tile = lt.tile * 256; tile < n; tile += lt.tiles * 256) {
    const int i = tile + tid;
    unsigned long long k = a.drop_key;
    bool head = false;
    if (i < n) {
      k = key[i];
      head = k != a.drop_key && (i == 0 || key[i - 1] != k);
    }
    int x = head ? 1 : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    int add = a.tile_heads[tile_slot(a.seg_base, l, 0, tile >> 8)];
    for (int w = 0; w < warp; ++w) add += warp_sum[w];
    if (head) {
      const int slot = add + x - 1;
      int q = i, plo = 0x7fffffff, phi = -1;
      for (; q < n && key[q] == k; ++q) {
        const int s = a.b.out_src[e0 + (int)idx[q]];
        const int lo = a.b.band_lo[s];
        const int hi = lo + (int)(a.b.band_off[s + 1] - a.b.band_off[s]);
        plo = min(plo, lo);
        phi = max(phi, hi);
        a.q_group[e0 + q] = slot;
      }
      a.g_word[e0 + slot] = (int32_t)k;
      a.g_start[e0 + slot] = i;
      a.g_len[e0 + slot] = q - i;
      a.g_plo[e0 + slot] = plo;
      a.g_phi[e0 + slot] = phi;
      a.g_celloff[e0 + slot] = phi - plo;  // scanned in place by k_pos_cell_offsets
    }
    __syncthreads();
  }
}

// One CTA per lattice: exclusive scan of the groups' cell counts (in place) + lattice total
__global__ void __launch_bounds__(256) k_pos_cell_offsets(PosArgs a) {
  __shared__ long long warp_sum[8];
  __shared__ long long carry_s;
  const int l = blockIdx.x;
  const int e0 = a.b.e_off[l], n = a.ngroups[l];
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = 0; tile < n; tile += 256) {
    const int i = tile + tid;
    const long long c = i < n ? a.g_celloff[e0 + i] : 0;
    const long long pre = cta_exclusive_scan<long long, 256>(c, warp_sum, carry_s);
    if (i < n) a.g_celloff[e0 + i] = (int32_t)min(pre, (long long)0x7fffffff);
  }
  if (tid == 0) a.lat_cells[l] = carry_s;
}

// grid (chunk lattices, tiles): per sorted arc the record the cell loop reads
__global__ void __launch_bounds__(256) k_pos_arcrec(PosArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = a.l0 + lt.l;
  const int n = a.seg_cnt[l];
  const int e0 = a.b.e_off[l];
  const unsigned long long* key = (a.where[l] ? a.key_b : a.key_a) + a.seg_base[l];
  const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + a.seg_base[l];
  ArcRec* rec = a.rec + (e0 - a.e_chunk0);
  for (int q = lt.tile * blockDim.x + threadIdx.x; q < n; q += lt.tiles * blockDim.x) {
    if (key[q] == a.drop_key) continue;
    const int e = e0 + (int)idx[q];
    const int4 r = a.b.out_rec[e];
    const int s = a.b.out_src[e];
    const int lo = a.b.band_lo[s];
    ArcRec rc;
    rc.base = a.b.band_off[s] - a.band_base - lo;
    rc.tail = __dadd_rn(-rec_cost(r, a.cp), 0.0);
    rc.beta = a.beta[r.x];
    rc.lo = lo;
    rc.hi = lo + (int)(a.b.band_off[s + 1] - a.b.band_off[s]);
    rec[q] = rc;
    if (a.arc_cellbase) {
      const int g = a.q_group[e0 + q];
      a.arc_cellbase[e] = a.cell_base[l] + a.g_celloff[e0 + g] - a.g_plo[e0 + g];
    }
  }
}

// grid (chunk lattices, tiles): group of the first cell of every 256-cell tile (one bisection per tile)
__global__ void __launch_bounds__(256) k_pos_tile_groups(PosArgs a) {
  const int l = a.l0 + blockIdx.x;
  const long long ncells = a.lat_cells[l];
  const int ng = a.ngroups[l];
  const int32_t* celloff = a.g_celloff + a.b.e_off[l];
  const long long ntiles = (ncells + 255) >> 8;
  for (long long t = (long long)blockIdx.y * blockDim.x + threadIdx.x; t < ntiles; t += (long long)gridDim.y * blockDim.x) {
    const long long first = t << 8;
    const int lo = last_le(celloff, 0, ng - 1, first);  // last group with celloff <= first
    a.tile_group[tile_slot(a.cell_base, l, a.l0, (int)t)] = lo;
  }
}

// grid (chunk lattices, tiles of 256 cells): one thread per (word, position) cell
__global__ void __launch_bounds__(256) k_pos_cells(PosArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = a.l0 + lt.l;
  const long long ncells = a.lat_cells[l];
  const int e0 = a.b.e_off[l];
  const int ng = a.ngroups[l];
  const int32_t* celloff = a.g_celloff + e0;
  const ArcRec* rec = a.rec + (e0 - a.e_chunk0);
  const int64_t cbase = a.cell_base[l];
  const double norm = a.tool == KLU_BEST_PATH2 ? a.beta[a.b.s_off[l]] : a.total[l];
  for (long long tile = (long long)lt.tile * 256; tile < ncells; tile += (long long)lt.tiles * 256) {
    const long long cell = tile + threadIdx.x;
    int g = a.tile_group[tile_slot(a.cell_base, l, a.l0, (int)(tile >> 8))];  // the lanes walk on from the tile's first group
    bool exists = false;
    if (cell < ncells) {
      while (g + 1 < ng && (long long)celloff[g + 1] <= cell) ++g;
      const int pos = a.g_plo[e0 + g] + (int)(cell - celloff[g]);
      const int q0 = a.g_start[e0 + g], q1 = q0 + a.g_len[e0 + g];
      const bool plain = a.tool != KLU_POSITION;
      // fw[(len, s)] + arc_lkh + bw[next] (position tool, :162-163); fw[u] + bw[v] - cost
      // (best-path2 :134, position-post :111-113); -inf when the arc's source does not hold `pos`
      auto fw = [&](const ArcRec& rc) -> double {  // -inf: (length, state) is not a state of the unfolded lattice
        return (pos >= rc.lo && pos < rc.hi) ? a.alpha2[rc.base + pos] : neg_inf();
      };
      auto term = [&](const ArcRec& rc, double al) -> double {
        return plain ? __dadd_rn(__dadd_rn(al, rc.beta), rc.tail) : __dadd_rn(__dadd_rn(al, rc.tail), rc.beta);
      };
      // Pass 1 (no loop-carried chain beyond a compare): maximum, number of finite terms, the
      // first two of them, the best single arc.
      double bestv = neg_inf();  // the best single term: also the maximum the sum is taken around
      int nterm = 0, besta = -1;
#pragma unroll 2
      for (int q = q0; q < q1; ++q) {
        const ArcRec rc = rec[q];
        const double al = fw(rc);
        const double v = term(rc, al);
        if (!(al > neg_inf())) continue;
        nterm += v > neg_inf() ? 1 : 0;
        if (besta < 0 || v > bestv) {
          // strict '>' in the reference's iteration order (input state, arc order):
          // kwsbin2/lattice-word-index-position.cc:178
          bestv = v;
          besta = q;
        } else if (a.tool == KLU_POSITION && v == bestv) {
          const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + a.seg_base[l];
          if (a.b.out_orig[e0 + (int)idx[q]] < a.b.out_orig[e0 + (int)idx[besta]]) besta = q;
        }
      }
      exists = besta >= 0;
      const double m = bestv;
      if (exists) {
        double sum;
        if (nterm >= 3) {
          // Pass 2: exp terms into two accumulators (exp(-inf) = 0 for the arcs that do not reach)
          double s0 = 0.0, s1 = 0.0;
          int q = q0;
          for (; q + 1 < q1; q += 2) {
            const ArcRec ra = rec[q], rb = rec[q + 1];
            const double va = term(ra, fw(ra)), vb = term(rb, fw(rb));
            s0 += fast_exp(va - m);
            s1 += fast_exp(vb - m);
          }
          if (q < q1) {
            const ArcRec ra = rec[q];
            s0 += fast_exp(term(ra, fw(ra)) - m);
          }
          sum = m + fast_log(s0 + s1);
        } else {  // one or two terms: Kaldi's LogAdd exactly
          sum = neg_inf();
          for (int q = q0; q < q1; ++q) {
            const ArcRec rc = rec[q];
            sum = log_add(sum, term(rc, fw(rc)));
          }
        }
        const unsigned int word = (unsigned int)a.g_word[e0 + g];
        if (a.tool == KLU_BEST_PATH2) {
          // latbin/lattice-best-path2.cc:145-147,175: posterior clamped to <= 0, float cost 1 - P
          const double post = fmin(0.0, sum - norm);
          double ls;  // LogSub(0, post) [ext]
          if (post >= 0.0) ls = neg_inf();
          else {
            ls = log(1.0 - exp(post));
            if (ls != ls) ls = neg_inf();
          }
          a.ccost[cbase + cell] = (double)(float)exp(ls);
        } else {
          CellRec cr;
          cr.val = sum - norm;
          cr.exists = 1u;
          cr.pad = 0u;
          if (a.tool == KLU_POSITION_POST) {
            cr.key = ((unsigned long long)(pos + 1) << a.bits_label) | word;
            cr.t0 = cr.t1 = 0;
          } else {
            const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + a.seg_base[l];
            const int e = e0 + (int)idx[besta];
            cr.key = ((unsigned long long)word << a.bits_len) | (unsigned long long)pos;
            cr.t0 = a.b.time[a.b.out_src[e]];
            cr.t1 = a.b.time[a.b.out_rec[e].x];
          }
          a.cell[cbase + cell] = cr;
        }
      }
      if (!exists && a.tool != KLU_BEST_PATH2) {
        CellRec cr;
        cr.val = 0.0;
        cr.key = 0ULL;
        cr.t0 = cr.t1 = 0;
        cr.exists = 0u;
        cr.pad = 0u;
        a.cell[cbase + cell] = cr;
      }
    }
    if (a.tool != KLU_BEST_PATH2) {
      const int cnt = __syncthreads_count(exists);
      if (threadIdx.x == 0) a.ctile[tile_slot(a.cell_base, l, a.l0, (int)(tile >> 8))] = cnt;
    }
  }
}

// grid (chunk lattices, tiles): existing cells -> (order key, cell) pairs, densely
__global__ void __launch_bounds__(256) k_pos_compact(PosArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  __shared__ int warp_sum[8];
  const int l = a.l0 + lt.l;
  const long long ncells = a.lat_cells[l];
  const int64_t cbase = a.cell_base[l];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (long long tile = (long long)lt.tile * 256; tile < ncells; tile += (long long)lt.tiles * 256) {
    const long long cell = tile + tid;
    CellRec cr;
    cr.exists = 0u;
    if (cell < ncells) cr = a.cell[cbase + cell];
    const bool exists = cr.exists != 0u;
    int x = exists ? 1 : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    int add = a.ctile[tile_slot(a.cell_base, l, a.l0, (int)(tile >> 8))];
    for (int w = 0; w < warp; ++w) add += warp_sum[w];
    if (exists) {
      const int slot = add + x - 1;
      const double logp = cr.val + 0.0;  // -0.0 and +0.0 compare equal in the reference's sort
      if (a.tool == KLU_POSITION_POST) {
        const float f = (float)logp + 0.0f;
        a.key2[cbase + slot] = ((cr.key >> a.bits_label) << 32) | (unsigned long long)(~ord_f32(f));
      } else {
        a.key32[cbase + slot] = (unsigned int)((~ord_f64(logp)) >> 32);
      }
      a.idx2[cbase + slot] = (unsigned int)cell;
    }
    __syncthreads();
  }
}

// The order sort of the position index runs on the high half of the f64 keys only (32-bit
// keys: a third less traffic per pass); runs that agree there (log-posteriors equal to ~1e-6
// relative: a handful per lattice) are settled here by a stable insertion sort on the full
// key, read back from the cell values, one thread per run.
struct PosFixArgs {
  const int64_t* seg_base;
  const int32_t* seg_cnt;
  const unsigned char* where;
  unsigned int *key_a, *key_b;
  unsigned int *val_a, *val_b;
  const CellRec* cell;
  int l0;
};

__global__ void __launch_bounds__(256) k_pos_order_fixup(PosFixArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = a.l0 + lt.l;
  const int n = a.seg_cnt[l];
  const int64_t base = a.seg_base[l];
  const unsigned int* K = (a.where[lt.l] ? a.key_b : a.key_a) + base;
  unsigned int* V = (a.where[lt.l] ? a.val_b : a.val_a) + base;
  const CellRec* cv = a.cell + base;
  for (int i = lt.tile * blockDim.x + threadIdx.x; i + 1 < n; i += lt.tiles * blockDim.x) {
    const unsigned int t = K[i];
    if ((i > 0 && K[i - 1] == t) || K[i + 1] != t) continue;  // not the head of a run
    int j = i + 1;
    while (j < n && K[j] == t) {  // insert element j into the ordered [i, j)
      const unsigned int v = V[j];
      const unsigned long long k = ~ord_f64(cv[v].val + 0.0);
      int q = j;
      while (q > i && (~ord_f64(cv[V[q - 1]].val + 0.0)) > k) {
        V[q] = V[q - 1];
        --q;
      }
      V[q] = v;
      ++j;
    }
  }
}

struct PosGatherArgs {
  PosArgs p;
  const int64_t* res_off;
  const unsigned char* where2;  // chunk-local: which order-sort buffer holds lattice l0 + i
  const unsigned int *idx2_a, *idx2_b;
  int32_t *c0, *c1, *c2, *c3;
  double* v;
  float* vf;
};

// grid (chunk lattices, tiles): output row i of a lattice = its i-th cell in log-posterior order
__global__ void __launch_bounds__(256) k_pos_gather(PosGatherArgs g) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const PosArgs& a = g.p;
  const int l = a.l0 + lt.l;
  const int n = a.rcnt[l];
  const int64_t cbase = a.cell_base[l];
  const int64_t out = g.res_off[l];
  const unsigned int* ord = (g.where2[lt.l] ? g.idx2_b : g.idx2_a) + cbase;
  for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
    const CellRec cr = a.cell[cbase + ord[i]];  // the one scattered read of a row
    if (a.tool == KLU_POSITION) {
      const unsigned long long lm = (1ULL << a.bits_len) - 1ULL;
      g.c0[out + i] = (int32_t)(cr.key >> a.bits_len);
      g.c1[out + i] = (int32_t)(cr.key & lm) + 1;  // 1-based position, :107
      g.c2[out + i] = cr.t0;
      g.c3[out + i] = cr.t1;
      g.v[out + i] = cr.val;
    } else {  // position-post: (0-based position index, word, float)
      const unsigned long long lm = (1ULL << a.bits_label) - 1ULL;
      g.c0[out + i] = (int32_t)(cr.key >> a.bits_label) - 1;
      g.c1[out + i] = (int32_t)(cr.key & lm);
      g.vf[out + i] = (float)cr.val;
    }
  }
}

int bits_for(int64_t maxv) {
  int b = 1;
  while (b < 63 && ((int64_t)1 << b) <= maxv) ++b;
  return b;
}

}  // namespace

int run_position_tool(klu_ctx* c, int tool, const klu_opts* o) {
  const int32_t L = c->L;
  if (tool != KLU_POSITION_POST)  // best-path2 reports frames (:102), the index carries segments
    for (int32_t l = 0; l < L; ++l)
      if (!c->h_times_ok[l]) {
        // CompactLatticeStateTimes [ext] KALDI_ASSERTs on this
        set_error("lattice " + std::to_string(l) + ": inconsistent state times (lattice is not aligned)");
        return 1;
      }
  const bool use_beam = tool == KLU_POSITION && o->beam != INFINITY;
  if (use_beam && !(o->beam > 0.0f)) {
    set_error("--beam must be positive");  // KALDI_ASSERT(beam > 0.0) in PruneLattice [ext]
    return 1;
  }
  const CostParams cp = make_cost_params(o, false);
  if (use_beam) KLU_TRY(run_tropical_sweeps(c, cp));
  KLU_TRY(run_log_sweeps(c, cp, use_beam, o->beam));
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = 0;
  KLU_TRY(c->d_res[5].reserve(sizeof(int64_t) * (L + 1)));
  KLU_CUDA(cudaMemsetAsync(c->d_res[5].p, 0, sizeof(int64_t) * (L + 1), c->stream));
  if (L == 0 || c->E == 0) {
    if (tool == KLU_BEST_PATH2 && L > 0) {  // lattices without arcs still report a (possibly empty) path
      BestPathChunk ch;
      ch.l0 = 0;
      ch.l1 = L;
      ch.band_base = 0;
      KLU_TRY(run_banded_alpha(c, cp, false, 0.f, 0, L));
      ch.alpha2 = c->d_alpha2.as<double>();
      ch.arc_cellbase = nullptr;
      ch.ecost = nullptr;
      ch.first_chunk = true;
      KLU_TRY(best_path2_decode(c, cp, ch));
    }
    c->last_entries = -1;
    return 0;
  }
  const size_t E1 = (size_t)c->E;
  enum { P_SEG = 0, P_KEYA, P_KEYB, P_IDXA, P_IDXB, P_GROUPS, P_LATMETA, P_REC, P_CELL, P_ORDER, P_TILES, P_CTILES };
  DevBuf* sc = c->d_scratch;
  // ---- per-lattice metadata: seg_base (int64 L+1) | seg_cnt (int32 L) | where (2L bytes)
  KLU_TRY(sc[P_SEG].reserve(8 * (size_t)(L + 1) + 4 * (size_t)L + 2 * (size_t)L + 64));
  int64_t* d_seg_base = sc[P_SEG].as<int64_t>();
  int32_t* d_seg_cnt = reinterpret_cast<int32_t*>(d_seg_base + L + 1);
  unsigned char* d_where = reinterpret_cast<unsigned char*>(d_seg_cnt + L);
  std::vector<int32_t> seg_cnt(L);
  for (int32_t l = 0; l < L; ++l) seg_cnt[l] = (int32_t)(c->h_e_off[l + 1] - c->h_e_off[l]);
  KLU_CUDA(cudaMemcpyAsync(d_seg_base, c->h_e_off.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemcpyAsync(d_seg_cnt, seg_cnt.data(), 4 * (size_t)L, cudaMemcpyHostToDevice, c->stream));
  KLU_TRY(sc[P_KEYA].reserve(8 * E1));
  KLU_TRY(sc[P_KEYB].reserve(8 * E1));
  KLU_TRY(sc[P_IDXA].reserve(4 * E1));
  KLU_TRY(sc[P_IDXB].reserve(4 * E1));
  // groups: word, start, len, plo, phi, celloff, q_group (int32 x E each) + arc_cellbase (int64 x E)
  KLU_TRY(sc[P_GROUPS].reserve(4 * 7 * E1 + 8 * E1 + 64));
  // ngroups (int32 L) | rcnt (int32 L) | lat_cells (int64 L) | cell_base (int64 L+1)
  KLU_TRY(sc[P_LATMETA].reserve(8 * (size_t)L + 8 * (size_t)L + 8 * (size_t)(L + 1) + 64));
  KLU_TRY(sc[P_TILES].reserve(4 * ((E1 >> 8) + (size_t)L + 2)));

  int fmode = 0, fn = 0;
  if (tool == KLU_POSITION) KLU_TRY(upload_filter(c, o, &fmode, &fn));

  PosArgs a;
  memset(&a, 0, sizeof(a));
  a.b = c->view();
  a.cp = make_cost_params(o, tool == KLU_POSITION_POST);  // position-post adds g + a in float
  a.tool = tool;
  a.filter_mode = fmode;
  a.filter_n = fn;
  a.filter = c->d_filter.as<int32_t>();
  a.beta = c->d_beta.as<double>();
  a.total = c->d_total.as<double>();
  a.use_beam = use_beam ? 1 : 0;
  a.vfwd = c->d_vfwd.as<double>();
  a.vbwd = c->d_vbwd.as<double>();
  a.best = c->d_best.as<double>();
  a.beam = (double)o->beam;
  a.bits_label = bits_for(c->max_label);
  a.bits_len = bits_for(c->max_len);
  if (a.bits_label + a.bits_len + 1 > 62 || a.bits_len > 30) {
    set_error("index key does not fit 62 bits (labels/times too large)");
    return 1;
  }
  a.drop_key = 1ULL << a.bits_label;
  a.seg_base = d_seg_base;
  a.seg_cnt = d_seg_cnt;
  a.key_a = sc[P_KEYA].as<unsigned long long>();
  a.key_b = sc[P_KEYB].as<unsigned long long>();
  a.idx_a = sc[P_IDXA].as<unsigned int>();
  a.idx_b = sc[P_IDXB].as<unsigned int>();
  a.where = d_where;
  a.tile_heads = sc[P_TILES].as<int32_t>();
  int32_t* gp = sc[P_GROUPS].as<int32_t>();
  a.g_word = gp;
  a.g_start = gp + E1;
  a.g_len = gp + 2 * E1;
  a.g_plo = gp + 3 * E1;
  a.g_phi = gp + 4 * E1;
  a.g_celloff = gp + 5 * E1;
  a.q_group = gp + 6 * E1;
  long long* d_arc_cellbase = reinterpret_cast<long long*>(gp + 7 * E1 + (E1 & 1));
  a.ngroups = sc[P_LATMETA].as<int32_t>();
  a.rcnt = a.ngroups + L;
  a.lat_cells = reinterpret_cast<long long*>(a.rcnt + L);
  int64_t* d_cell_base = reinterpret_cast<int64_t*>(a.lat_cells + L);
  a.cell_base = d_cell_base;

  int64_t max_arcs = 0;
  for (int32_t l = 0; l < L; ++l) max_arcs = std::max<int64_t>(max_arcs, seg_cnt[l]);
  const int arc_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  const int arc_tiles_full = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 8192));
  // ---- arcs grouped by word
  {
    KLU_LAUNCH(c, "k_pos_keys");
    k_pos_keys<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_pos_keys"));
  SegSortArgs s1;
  s1.seg_base = d_seg_base;
  s1.seg_cnt = d_seg_cnt;
  s1.key_a = a.key_a;
  s1.val_a = a.idx_a;
  s1.key_b = a.key_b;
  s1.val_b = a.idx_b;
  s1.where = d_where;
  s1.lo_bit = 0;
  s1.hi_bit = a.bits_label + 1;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, s1, L, c->E));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(words)"));
  {
    KLU_LAUNCH(c, "k_pos_head_count");
    k_pos_head_count<<<dim3(L, arc_tiles_full), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_pos_head_count"));
  {
    KLU_LAUNCH(c, "k_tile_prefix");
    k_tile_prefix<<<L, 256, 0, c->stream>>>(d_seg_base, nullptr, d_seg_cnt, 0, a.tile_heads, a.ngroups);
  }
  KLU_TRY(check_launch("k_tile_prefix(groups)"));
  {
    KLU_LAUNCH(c, "k_pos_groups");
    k_pos_groups<<<dim3(L, arc_tiles_full), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_pos_groups"));
  {
    KLU_LAUNCH(c, "k_pos_cell_offsets");
    k_pos_cell_offsets<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_pos_cell_offsets"));
  // ---- the one host round trip: cells per lattice (chunk plan and scratch sizes depend on it)
  std::vector<long long> lat_cells(L);
  KLU_CUDA(cudaMemcpyAsync(lat_cells.data(), a.lat_cells, 8 * (size_t)L, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  for (int32_t l = 0; l < L; ++l)
    if (lat_cells[l] >= ((long long)1 << 31)) {
      set_error("lattice " + std::to_string(l) + ": more than 2^31 (word, position) cells");
      return 1;
    }
  // ---- chunk plan: contiguous lattice ranges whose cells (56 B each) and bands (8 B per cell) fit
  int64_t cell_budget = (int64_t)1 << 28;
  {
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
      size_t held = sc[P_REC].cap + sc[P_CELL].cap + sc[P_ORDER].cap + sc[P_CTILES].cap;
      const int64_t fit = (int64_t)((free_b + held) / 3 / 56);
      cell_budget = std::min<int64_t>((int64_t)1 << 31, std::max<int64_t>((int64_t)1 << 24, fit));
    }
  }
  if (const char* env = getenv("KLU_ENTRY_BUDGET")) cell_budget = std::max<long long>(1, atoll(env));  // tests
  const int64_t band_budget = getenv("KLU_ENTRY_BUDGET") ? cell_budget : (int64_t)1 << 30;
  std::vector<int64_t> cell_base(L + 1, 0);
  std::vector<int32_t> chunk_first(1, 0);
  {
    int64_t acc = 0, band_acc = 0;
    for (int32_t l = 0; l < L; ++l) {
      const int64_t band = c->h_band_off[l + 1] - c->h_band_off[l];
      if (l > chunk_first.back() && (acc + lat_cells[l] > cell_budget || band_acc + band > band_budget)) {
        chunk_first.push_back(l);
        acc = 0;
        band_acc = 0;
      }
      cell_base[l] = acc;
      acc += lat_cells[l];
      band_acc += band;
    }
    chunk_first.push_back(L);
  }
  int64_t N = 1, max_chunk_arcs = 1;  // largest chunk in cells / in arcs
  for (size_t k = 0; k + 1 < chunk_first.size(); ++k) {
    const int32_t last = chunk_first[k + 1] - 1;
    N = std::max<int64_t>(N, cell_base[last] + lat_cells[last]);
    max_chunk_arcs = std::max<int64_t>(max_chunk_arcs, c->h_e_off[last + 1] - c->h_e_off[chunk_first[k]]);
  }
  KLU_CUDA(cudaMemcpyAsync(d_cell_base, cell_base.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_TRY(sc[P_REC].reserve(sizeof(ArcRec) * (size_t)max_chunk_arcs));
  const bool bp2 = tool == KLU_BEST_PATH2;
  KLU_TRY(sc[P_CELL].reserve((bp2 ? 8 : sizeof(CellRec)) * (size_t)N + 64));
  if (!bp2) {
    KLU_TRY(sc[P_ORDER].reserve(24 * (size_t)N + 64));
  }
  KLU_TRY(sc[P_CTILES].reserve(8 * (((size_t)N >> 8) + (size_t)L + 2)));
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // cell_base is a stack object
  a.rec = sc[P_REC].as<ArcRec>();
  a.cell = sc[P_CELL].as<CellRec>();
  a.ccost = sc[P_CELL].as<double>();
  unsigned long long* key2_a = sc[P_ORDER].as<unsigned long long>();
  unsigned long long* key2_b = key2_a + N;
  unsigned int* idx2_a = reinterpret_cast<unsigned int*>(key2_b + N);
  unsigned int* idx2_b = idx2_a + N;
  unsigned int* key32_a = reinterpret_cast<unsigned int*>(key2_a);  // the position index sorts 32-bit keys
  unsigned int* key32_b = reinterpret_cast<unsigned int*>(key2_b);
  a.key2 = key2_a;
  a.key32 = key32_a;
  a.idx2 = idx2_a;
  a.ctile = sc[P_CTILES].as<int32_t>();
  a.tile_group = a.ctile + (((size_t)N >> 8) + (size_t)L + 2);
  a.arc_cellbase = bp2 ? d_arc_cellbase : nullptr;

  int64_t res_cap = 0, res_used = 0;
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
    a.band_base = c->h_band_off[l0];
    a.e_chunk0 = (int)c->h_e_off[l0];
    KLU_TRY(run_banded_alpha(c, cp, use_beam, o->beam, l0, l1));
    a.alpha2 = c->d_alpha2.as<double>();
    int64_t chunk_max_arcs = 0, chunk_max_cells = 1;
    for (int32_t l = l0; l < l1; ++l) {
      chunk_max_arcs = std::max<int64_t>(chunk_max_arcs, seg_cnt[l]);
      chunk_max_cells = std::max<int64_t>(chunk_max_cells, lat_cells[l]);
    }
    const int tiles = (int)std::max<int64_t>(1, std::min<int64_t>((chunk_max_arcs + 255) / 256, 64));
    const int ctiles = (int)std::max<int64_t>(1, std::min<int64_t>((chunk_max_cells + 255) / 256, 16384));
    {
      KLU_LAUNCH(c, "k_pos_arcrec");
      k_pos_arcrec<<<dim3(nl, tiles), 256, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_pos_arcrec"));
    {
      KLU_LAUNCH(c, "k_pos_tile_groups");
      k_pos_tile_groups<<<dim3(nl, (unsigned)std::max<int64_t>(1, std::min<int64_t>(((chunk_max_cells >> 8) + 256) / 256, 64))), 256, 0,
                          c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_pos_tile_groups"));
    {
      KLU_LAUNCH(c, "k_pos_cells");
      k_pos_cells<<<dim3(nl, ctiles), 256, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_pos_cells"));
    if (bp2) {
      BestPathChunk ch;
      ch.l0 = l0;
      ch.l1 = l1;
      ch.band_base = a.band_base;
      ch.alpha2 = a.alpha2;
      ch.arc_cellbase = d_arc_cellbase;
      ch.ecost = a.ccost;
      ch.first_chunk = k == 0;
      KLU_TRY(best_path2_decode(c, cp, ch));
      continue;
    }
    {
      KLU_LAUNCH(c, "k_tile_prefix");
      k_tile_prefix<<<nl, 256, 0, c->stream>>>(d_cell_base, a.lat_cells, nullptr, l0, a.ctile, a.rcnt);
    }
    KLU_TRY(check_launch("k_tile_prefix(cells)"));
    {
      KLU_LAUNCH(c, "k_pos_compact");
      k_pos_compact<<<dim3(nl, ctiles), 256, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_pos_compact"));
    unsigned char* where2 = d_where + L;  // chunk-local flags
    if (tool == KLU_POSITION) {
      SegSortArgs32 s2;
      s2.seg_base = d_cell_base + l0;
      s2.seg_cnt = a.rcnt + l0;
      s2.key_a = key32_a;
      s2.val_a = idx2_a;
      s2.key_b = key32_b;
      s2.val_b = idx2_b;
      s2.where = where2;
      s2.lo_bit = 0;
      s2.hi_bit = 32;
      {
        KLU_LAUNCH(c, "k_seg_radix_sort");
        KLU_TRY(seg_sort_launch(c, s2, nl, N));
      }
      KLU_TRY(check_launch("k_seg_radix_sort(order)"));
      PosFixArgs f;
      f.seg_base = d_cell_base;
      f.seg_cnt = a.rcnt;
      f.where = where2;
      f.key_a = key32_a, f.key_b = key32_b;
      f.val_a = idx2_a, f.val_b = idx2_b;
      f.cell = a.cell;
      f.l0 = l0;
      {
        KLU_LAUNCH(c, "k_order_fixup");
        k_pos_order_fixup<<<dim3(nl, ctiles), 256, 0, c->stream>>>(f);
      }
      KLU_TRY(check_launch("k_order_fixup"));
    } else {
      SegSortArgs s2;
      s2.seg_base = d_cell_base + l0;
      s2.seg_cnt = a.rcnt + l0;
      s2.key_a = key2_a;
      s2.val_a = idx2_a;
      s2.key_b = key2_b;
      s2.val_b = idx2_b;
      s2.where = where2;
      s2.lo_bit = 0;
      s2.hi_bit = 64;
      {
        KLU_LAUNCH(c, "k_seg_radix_sort");
        KLU_TRY(seg_sort_launch(c, s2, nl, N));
      }
      KLU_TRY(check_launch("k_seg_radix_sort(order)"));
    }
    KLU_TRY(scan_counts(c, a.rcnt, l0, l1, c->d_res[5].as<int64_t>(), "k_scan_counts"));
    {
      int64_t upto = 0;
      KLU_CUDA(cudaMemcpyAsync(&upto, c->d_res[5].as<int64_t>() + l1, sizeof(int64_t), cudaMemcpyDeviceToHost,
                               c->stream));
      KLU_CUDA(cudaStreamSynchronize(c->stream));
      KLU_TRY(grow_results(upto));
      res_used = upto;
    }
    PosGatherArgs g;
    g.p = a;
    g.res_off = c->d_res[5].as<int64_t>();
    g.where2 = where2;
    g.idx2_a = idx2_a;
    g.idx2_b = idx2_b;
    g.c0 = c->d_res[0].as<int32_t>();
    g.c1 = c->d_res[1].as<int32_t>();
    g.c2 = c->d_res[2].as<int32_t>();
    g.c3 = c->d_res[3].as<int32_t>();
    g.v = c->d_res[4].as<double>();
    g.vf = c->d_res[4].as<float>();
    {
      KLU_LAUNCH(c, "k_pos_gather");
      k_pos_gather<<<dim3(nl, ctiles), 256, 0, c->stream>>>(g);
    }
    KLU_TRY(check_launch("k_pos_gather"));
  }
  c->last_entries = -1;  // known after klu_result_offsets()
  return 0;
}

}  // namespace klu
