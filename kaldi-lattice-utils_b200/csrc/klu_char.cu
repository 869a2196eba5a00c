// klu_char.cu -- lattice-char-index-position on the device.
//
// Reference: kwsbin2/lattice-char-index-position.cc:137-284 with kwsbin2/utils.h:41-303
// and fstext/fstext-utils2.h:278-603 -- an OpenFst pipeline (state splitting by label
// group and word count, GroupFactorFst, RmEpsilon, two determinisations, compose,
// n-best).  Its net semantics (SURVEY.md 8a C1-C6, Appendix B.4): every maximal run
// of same-group (non-whitespace, non-epsilon) arcs along any path is a pseudo-word;
// runs are keyed by (word position, label sequence); a key's score is
//   log sum over its runs of  fw[u] * w(run) * exit(x)  -  total,
// its segment (t0, t1) that of the single best run; the n best keys are kept.
//
// Device formulation (no FST is materialised):
//   1. log backward sweep (beta, total = beta[start]) -- klu_sweep.cu;
//   2. word-count bands per state (integer level sweep), then the forward scores of
//      the split lattice A[state][count][incoming group] (level-synchronous DP);
//   3. exit weights exit[state][group];
//   4. frontier determinisation: items (trie node, state, log-sum weight, best single
//      weight + its t0).  Depth 0 = every (split state, entering arc); each round
//      accumulates the node scores, expands every item along its same-group arcs,
//      and merges equal (node, label, state) candidates with a per-lattice stable
//      radix sort + segmented LogAdd (new trie nodes = runs of equal (node, label));
//   5. rows = nodes with a finite score; per-lattice n-best by two stable sorts;
//      label sequences by walking the trie; the final (logp desc, string asc, pos
//      asc) order of the <= nbest rows is applied on the host at fetch time.
#include <limits.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

constexpr int kKeyStateBits = 20, kKeyCharBits = 20, kKeyParentBits = 24;

struct CharArgs {
  BatchView b;
  CostParams cp;
  const int32_t* glabels;  // sorted labels with an explicit group
  const int32_t* gdense;   // their dense group index
  int ngl, NG, dflt;       // #explicit labels, #dense groups, dense index of the default group
  unsigned int inc_mask, del_mask;
  int eps;                 // dense index of group 0 (epsilon)
  int segment;             // lattice-char-index-segment: keys carry frame tags instead of word counts
  int use_beam;
  const double *vfwd, *vbwd, *best;
  double beam;
  const double* beta;
  int32_t *nlo, *nhi;          // [S] word-count band per state
  int32_t* cell_cnt;           // [S] cells per state (band width * NG)
  const int32_t* cell_loc;     // [S] lattice-local first cell
  const int64_t* cell_base;    // [L] first cell of each lattice
  double* A;                   // split forward scores
  double* exitw;               // [S * NG]
  double* cont;                // [S * NG] in-group continuation mass C (k_char_cont)
};

__device__ __forceinline__ int group_of(const CharArgs& a, int label) {
  int lo = 0, hi = a.ngl - 1;
  while (lo <= hi) {
    const int mid = (lo + hi) >> 1;
    const int v = a.glabels[mid];
    if (v == label) return a.gdense[mid];
    if (v < label) lo = mid + 1;
    else hi = mid - 1;
  }
  return a.dflt;
}

__device__ __forceinline__ bool char_arc_pruned(const CharArgs& a, int l, int src, int dst, const int4& r) {
  if (!a.use_beam) return false;
  CostParams cp = a.cp;
  cp.float_sum = 0;
  const double fb = __dadd_rn(a.vfwd[src], __dadd_rn(rec_cost(r, cp), a.vbwd[dst]));
  return fb > __dadd_rn(a.best[l], a.beam);
}

__device__ __forceinline__ bool char_final_pruned(const CharArgs& a, int l, int s, double fcost) {
  if (!a.use_beam) return false;
  return __dadd_rn(fcost, a.vfwd[s]) > __dadd_rn(a.best[l], a.beam) && fcost != pos_inf();
}

// ---- generic per-lattice exclusive scan: one CTA per lattice ---------------------
// elements of lattice l: [beg(l), beg(l) + n(l)); out_loc[i] = exclusive prefix inside
// the lattice, tot[l] = lattice total
struct SegRange {
  const int32_t* off32;   // begin = off32[l], n = off32[l+1] - off32[l]   (or)
  const int64_t* base64;  // begin = base64[l], n = cnt32[l]
  const int32_t* cnt32;
};
__device__ __forceinline__ void seg_range(const SegRange& r, int l, int64_t* beg, int* n) {
  if (r.off32) {
    *beg = r.off32[l];
    *n = r.off32[l + 1] - r.off32[l];
  } else {
    *beg = r.base64[l];
    *n = r.cnt32[l];
  }
}

__global__ void __launch_bounds__(256) k_char_scan(SegRange rg, const int32_t* cnt, int32_t* out_loc, long long* tot) {
  __shared__ long long warp_sum[8];
  __shared__ long long carry_s;
  const int l = blockIdx.x;
  int64_t beg;
  int n;
  seg_range(rg, l, &beg, &n);
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = 0; tile < n; tile += 1024) {  // four consecutive elements per thread
    const int i0 = tile + tid * 4;
    int cc[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) cc[q] = i0 + q < n ? cnt[beg + i0 + q] : 0;
    const long long c = (long long)cc[0] + cc[1] + cc[2] + cc[3];
    long long run = cta_exclusive_scan<long long, 256>(c, warp_sum, carry_s);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (i0 + q < n) out_loc[beg + i0 + q] = (int32_t)run;
      run += cc[q];
    }
  }
  if (tid == 0) tot[l] = carry_s;
}

// ---- 2a. word-count bands: one warp per lattice, level by level -------------------
__global__ void __launch_bounds__(128) k_char_bands(CharArgs a) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const BatchView& b = a.b;
  if (warp >= b.L) return;
  const int l = warp;
  const int s0 = b.s_off[l], s1 = b.s_off[l + 1];
  if (s0 == s1) return;
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  for (int s = lv[0] + lane; s < lv[1]; s += 32) {
    a.nlo[s] = s == s0 ? 0 : INT_MAX;
    a.nhi[s] = s == s0 ? 0 : -1;
  }
  __syncwarp();
  for (int j = 1; j < nl; ++j) {
    for (int s = lv[j] + lane; s < lv[j + 1]; s += 32) {
      int lo = INT_MAX, hi = -1;
      for (int e = b.in_off[s]; e < b.in_off[s + 1]; ++e) {
        const int4 r = b.in_rec[e];
        const int plo = a.nlo[r.x], phi = a.nhi[r.x];
        if (phi < plo) continue;  // unreachable source
        const int inc = (a.inc_mask >> group_of(a, r.w)) & 1u;
        lo = min(lo, plo);
        hi = max(hi, phi + inc);
      }
      a.nlo[s] = lo;
      a.nhi[s] = hi;
    }
    __syncwarp();
  }
  for (int s = s0 + lane; s < s1; s += 32) {
    const int w = a.nhi[s] >= a.nlo[s] ? a.nhi[s] - a.nlo[s] + 1 : 0;
    a.cell_cnt[s] = w * a.NG;
  }
}

__device__ __forceinline__ long long cell_of(const CharArgs& a, int l, int s) {
  return a.cell_base[l] + a.cell_loc[s];
}

// ---- 2b. forward scores of the split lattice --------------------------------------
// A[s][n][g] = log-sum of all paths start -> s whose last arc has group g and which
// crossed n word-counting group boundaries (fstext/fstext-utils2.h:413-513: a
// transition into group vg from a different group ug counts when vg is a counting
// group).  One CTA per lattice; a thread owns one (state, n, g) cell of the level.
__global__ void __launch_bounds__(256) k_char_fwd(CharArgs a) {
  const int lane = threadIdx.x, nth = blockDim.x;
  const BatchView& b = a.b;
  const int l = blockIdx.x;
  const int s0 = b.s_off[l], s1 = b.s_off[l + 1];
  if (s0 == s1) return;
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  const int NG = a.NG;
  for (int s = lv[0] + lane; s < lv[1]; s += nth) {
    const long long c0 = cell_of(a, l, s);
    for (int q = 0; q < a.cell_cnt[s]; ++q) a.A[c0 + q] = (s == s0 && q == a.eps) ? 0.0 : neg_inf();
  }
  __syncthreads();
  for (int j = 1; j < nl; ++j) {
    const int a0 = lv[j], a1 = lv[j + 1];
    const int q0 = a.cell_loc[a0];
    const int q1 = a1 < s1 ? a.cell_loc[a1] : a.cell_loc[a1 - 1] + a.cell_cnt[a1 - 1];
    for (int q = q0 + lane; q < q1; q += nth) {
      const int s = last_le(a.cell_loc, a0, a1 - 1, q);  // last state of the level with cell_loc <= q
      const int rel = q - a.cell_loc[s];
      const int n = a.nlo[s] + rel / NG, g = rel % NG;
      const int inc = (a.inc_mask >> g) & 1u;
      double acc = neg_inf();
      for (int e = b.in_off[s]; e < b.in_off[s + 1]; ++e) {
        const int4 r = b.in_rec[e];
        if (group_of(a, r.w) != g) continue;
        const int u = r.x;
        const int ulo = a.nlo[u], uhi = a.nhi[u];
        if (uhi < ulo) continue;
        if (char_arc_pruned(a, l, u, s, r)) continue;
        const double cost = rec_cost(r, a.cp);
        const long long uc = cell_of(a, l, u);
        for (int gu = 0; gu < NG; ++gu) {
          const int nu = gu == g ? n : n - inc;
          if (nu < ulo || nu > uhi) continue;
          const double x = a.A[uc + (long long)(nu - ulo) * NG + gu];
          if (x > neg_inf()) acc = log_add(acc, x - cost);
        }
      }
      a.A[a.cell_base[l] + q] = acc;
    }
    __syncthreads();
  }
}

// ---- 3. exit weights ----------------------------------------------------------------
// exit[s][g] = LogAdd(-cost(final(s)), sum over arcs s -> y whose group differs from g
// of -cost + beta[y])  (what RmEpsilon folds into the final weight, fstext-utils2.h:558-585)
__global__ void __launch_bounds__(256) k_char_exit(CharArgs a) {
  const BatchView& b = a.b;
  const int l = blockIdx.x;
  const int s0 = b.s_off[l], ns = b.s_off[l + 1] - s0;
  for (int t = blockIdx.y * blockDim.x + threadIdx.x; t < ns * a.NG; t += gridDim.y * blockDim.x) {
    const int s = s0 + t / a.NG, g = t % a.NG;
    double e = neg_inf();
    {
      const double fc = final_cost(b.fin_g[s], b.fin_a[s], a.cp);
      if (fc < pos_inf() && !char_final_pruned(a, l, s, fc)) e = -fc;
    }
    for (int k = b.out_off[s]; k < b.out_off[s + 1]; ++k) {
      const int4 r = b.out_rec[k];
      if (group_of(a, r.w) == g) continue;
      if (char_arc_pruned(a, l, s, r.x, r)) continue;
      e = log_add(e, -rec_cost(r, a.cp) + a.beta[r.x]);
    }
    a.exitw[(long long)s * a.NG + g] = e;
  }
}

// ---- 3b. in-group continuation mass (the n-best cut, see "frontier cut" below) ------
// C[x][g] = LogAdd(exit[x][g], sum over arcs x -> y with group g that k_char_count / k_char_expand
// follow (same costs, same beam test) of -cost + C[y][g]): the log-sum of every way a pseudo-word
// of group g that has reached x can still go on and end.  The backward twin of k_char_fwd: one CTA
// per lattice, levels in descending order, a thread per (state, group) of the level.
__global__ void __launch_bounds__(256) k_char_cont(CharArgs a) {
  const BatchView& b = a.b;
  const int l = blockIdx.x;
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  const int NG = a.NG;
  for (int j = nl - 1; j >= 0; --j) {
    const int a0 = lv[j], a1 = lv[j + 1];
    for (int t = threadIdx.x; t < (a1 - a0) * NG; t += blockDim.x) {
      const int x = a0 + t / NG, g = t % NG;
      double acc = a.exitw[(long long)x * NG + g];
      for (int k = b.out_off[x]; k < b.out_off[x + 1]; ++k) {
        const int4 r = b.out_rec[k];
        if (group_of(a, r.w) != g || char_arc_pruned(a, l, x, r.x, r)) continue;
        const double y = a.cont[(long long)r.x * NG + g];
        if (y > neg_inf()) acc = log_add(acc, y - rec_cost(r, a.cp));
      }
      a.cont[(long long)x * NG + g] = acc;
    }
    __syncthreads();
  }
}

// ---- 4. frontier determinisation ---------------------------------------------------
struct Frontier {
  // items of the current depth: lattice l owns [ibase[l], ibase[l] + icnt[l])
  const int64_t* ibase;
  const int32_t* icnt;
  const int32_t* it_node;   // global node id
  const int32_t* it_state;  // packed global state
  const double *it_wsum, *it_wmax;
  const int32_t* it_t0;
  // trie nodes (global pool)
  int32_t *nd_parent, *nd_chr, *nd_cnt, *nd_grp, *nd_lat, *nd_t0, *nd_t1, *nd_len;
  double *nd_total, *nd_best;
  // candidates of the next depth: lattice l owns [cbase[l], cbase[l] + ccnt[l])
  const int64_t* cbase;
  int32_t* ccnt;
  int32_t* cand_cnt;        // per item / per arc: candidates it emits
  const int32_t* cand_loc;  // lattice-local exclusive scan of cand_cnt
  unsigned long long* ckey;
  unsigned int* cval;
  double *c_wsum, *c_wmax;
  int32_t* c_t0;
  int32_t* c_state;            // segment mode: lattice-local destination state of every candidate
  unsigned long long* c_main;  // segment mode: (parent | label | frame tag) of every candidate
  // sorted candidates
  const unsigned long long *key_a, *key_b;
  const unsigned int *val_a, *val_b;
  const unsigned char* where;
  // next items
  int32_t *n_node, *n_state, *n_t0;
  double *n_wsum, *n_wmax;
  int32_t* ncnt;            // [L] items of the next depth
  int32_t *tile_i, *tile_n;  // per tile of 256 sorted candidates: item / node heads (then: heads before it)
  int64_t node_pool_base;   // first pool slot of the depth being created
  int64_t parent_pool_base; // first pool slot of the current depth (parents)
  int depth;
  // n-best cut (see "frontier cut" below)
  double* nd_ub;            // per node: subtree bound U
  const double* tau;        // [L] cut threshold tau (log-probability); nullptr = no cut
  int32_t* tk_cnt;          // [L] keys in the lattice's threshold segment; nullptr = no keys gathered
  const int32_t* tk_keep;   // [L] of them carried over from the last depth
  const int64_t* tk_wbase;  // [L] threshold segment (work buffer)
  const int64_t* tk_tbase;  // [L] carried-over keys (top buffer)
  unsigned long long* tk_work;
  const unsigned long long* tk_top;
  unsigned long long* cut_cnt;  // KLU_CHAR_DEBUG: candidates cut at this depth (else nullptr)
};

// ---- frontier cut --------------------------------------------------------------------
// Only the nbest best rows (trie nodes) of a lattice are kept, so a prefix none of whose
// extensions can reach them need not be expanded.  Exact bound (items (p, x, wsum) of node p of
// group g, exit[x][g], nd_total(p) = log-sum over the items of wsum + exit, k_char_accum):
//   1. C[x][g] (k_char_cont) is the log-sum over every in-group continuation of x, along the very
//      arcs and costs that k_char_count / k_char_expand follow, ended by an exit.
//   2. U(p) = log-sum over ALL items of p (exit -inf included) of wsum + C[x][g].  Every sub-path
//      that spells p or a descendant q of p passes through exactly one item of p and goes on along
//      such arcs, so U(p) >= nd_total(q) for every q of p's subtree.  Position keys (word count)
//      and segment keys (frame tags) only split the sub-paths further; the bound holds for both.
//   3. tau_l = the nbest-th largest row log-probability (nd_total - beta[start], as k_char_rowkey
//      forms it) among the lattice's final nodes; -inf until there are nbest of them.  The nodes
//      of a depth are final once k_char_accum has folded them; tau only rises.
//   4. An item of a node with U(p) - beta[start] < tau_l - delta emits no candidates.  The node
//      itself stays a row candidate; it is below tau, so it is never selected.
//   5. Every node whose log-probability is >= the final tau survives (rounding is monotone, so
//      U >= total gives U - beta >= total - beta).  Survivors keep their order inside a lattice
//      (depth, then key order: removing emptied parents renumbers the rest monotonically), so the
//      two stable row sorts and k_char_select pick the same nodes, ties at the cut included.
//   6. delta absorbs rounding: U and the totals are f64 sums of the same terms taken in different
//      orders.  An add or log_add rounds within 2 ulp of its result, and an error passes through a
//      later log_add with a factor <= 1; every sum reaches a row through fewer than 2^31 such steps
//      (the batch's work-item limit), whose operands are bounded by M = 1 + |tau| + |beta[start]|.
//      So U and a total differ from their exact values by < 2 * 2^31 * 2^-51 * M = 2^-19 M;
//      delta = 2^-16 M is eight times that.  delta only keeps more, so it cannot change a result.
// With nbest at least the rows a lattice ends up with, tau stays -inf and nothing is cut.
// lattice-char-index-utterance runs the position frontier without counting groups (every split state
// has count 0, so a trie node is one string and nd_total = log E[N(v)] + beta[start], N(v) = runs
// spelling v on a path).  Its rows are the exact occurrence log-probabilities P(v) = P(N(v) >= 1)
// (k_char_occ), and tau is the nbest-th best of those found so far:
//   2'. P(v) <= E[N(v)] = exp(nd_total(v)) <= exp(U(p)) for every descendant v of p (step 2 needs no
//       position or segment key), so the test of step 4 still never cuts a node that reaches tau.
//   4'. k_char_occ computes P(v) only for final nodes with nd_total - beta[start] >= tau - delta; any
//       other node is below the final tau by step 2', gets no value and is never a row.
//   6'. The occurrence sum adds the same kinds of terms as nd_total and U: path costs (add) folded by
//       log_add, over the same arcs and exits, each reaching the value through fewer than 2^31 steps
//       (a DP cell is one of the batch's work items), so its rounding error obeys the same bound and
//       delta covers the comparison of a rounded P(v) with a rounded U or nd_total.
constexpr double kCutSlack = 1.0 / 65536.0;

__device__ __forceinline__ bool below_cut(double ub_logp, double tau, double beta0) {
  if (!(tau > neg_inf())) return false;
  if (tau == pos_inf()) return true;  // nbest 0: no row is selected
  return ub_logp < tau - kCutSlack * (1.0 + fabs(tau) + fabs(beta0));
}

// inverse of ~ord_f64: the log-probability of a threshold key
__device__ __forceinline__ double key_logp(unsigned long long k) {
  const unsigned long long u = ~k;
  return __longlong_as_double((long long)((u & 0x8000000000000000ULL) ? (u & 0x7fffffffffffffffULL) : ~u));
}

// lattice-char-index-segment: SymbolToPathSegmentationFst (kwsbin2/utils.h:251-303) keeps
// an output label on every arc that enters a state where the sub-path may stop (a final
// state of the factor FST = a state with an exit): the end frame of that arc, + 1.
__device__ __forceinline__ unsigned long long frame_tag(const CharArgs& a, int x, int g) {
  return a.exitw[(long long)x * a.NG + g] > neg_inf() ? (unsigned long long)(a.b.time[x] + 1) : 0ULL;
}

// depth 0: candidates per out-order arc = cells of the source whose group differs
__global__ void __launch_bounds__(256) k_char_count0(CharArgs a, Frontier f) {
  const BatchView& b = a.b;
  const int l = blockIdx.x;
  const int e0 = b.e_off[l], e1 = b.e_off[l + 1];
  for (int e = e0 + blockIdx.y * blockDim.x + threadIdx.x; e < e1; e += gridDim.y * blockDim.x) {
    const int4 r = b.out_rec[e];
    const int u = b.out_src[e];
    const int g = group_of(a, r.w);
    int c = 0;
    if (g != a.eps && !((a.del_mask >> g) & 1u) && a.nhi[u] >= a.nlo[u] && !char_arc_pruned(a, l, u, r.x, r)) {
      const long long uc = cell_of(a, l, u);
      const int w = a.nhi[u] - a.nlo[u] + 1;
      for (int q = 0; q < w * a.NG; ++q)
        if (q % a.NG != g && a.A[uc + q] > neg_inf()) ++c;
    }
    f.cand_cnt[e] = c;
  }
}

__global__ void __launch_bounds__(256) k_char_emit0(CharArgs a, Frontier f) {
  const BatchView& b = a.b;
  const int l = blockIdx.x;
  const int e0 = b.e_off[l], e1 = b.e_off[l + 1];
  const int64_t base = f.cbase[l];
  for (int e = e0 + blockIdx.y * blockDim.x + threadIdx.x; e < e1; e += gridDim.y * blockDim.x) {
    if (f.cand_cnt[e] == 0) continue;
    const int4 r = b.out_rec[e];
    const int u = b.out_src[e];
    const int g = group_of(a, r.w);
    const int inc = (a.inc_mask >> g) & 1u;
    const double cost = rec_cost(r, a.cp);
    const long long uc = cell_of(a, l, u);
    const int w = a.nhi[u] - a.nlo[u] + 1;
    int64_t o = base + f.cand_loc[e];
    for (int q = 0; q < w * a.NG; ++q) {
      if (q % a.NG == g) continue;
      const double x = a.A[uc + q];
      if (!(x > neg_inf())) continue;
      if (a.segment) {  // root = the sub-path's first frame; merged only with equal frame tags
        f.c_main[o] = ((unsigned long long)b.time[u] << (kKeyCharBits + kKeyStateBits)) |
                      ((unsigned long long)(unsigned int)r.w << kKeyStateBits) | frame_tag(a, r.x, g);
        f.c_state[o] = r.x - b.s_off[l];
        f.ckey[o] = (unsigned long long)(r.x - b.s_off[l]);
      } else {
        const unsigned long long count = (unsigned long long)(a.nlo[u] + q / a.NG + inc);
        f.ckey[o] = (count << (kKeyCharBits + kKeyStateBits)) | ((unsigned long long)(unsigned int)r.w << kKeyStateBits) |
                    (unsigned long long)(r.x - b.s_off[l]);
      }
      f.cval[o] = (unsigned int)(o - base);
      f.c_wsum[o] = x - cost;
      f.c_wmax[o] = x - cost;
      f.c_t0[o] = b.time[u];
      ++o;
    }
  }
}

// node scores of the current depth: the first item of every node folds the node's
// items (they are sorted by state) with their exit weights, and the subtree bound U.
// With the cut on, rows above tau go to the lattice's threshold segment, after the keys
// carried over from the last depth (copied here from the top buffer).
__global__ void __launch_bounds__(256) k_char_accum(CharArgs a, Frontier f) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = f.icnt[l];
  const int64_t base = f.ibase[l];
  const int lane = threadIdx.x & 31;
  const double beta0 = a.beta[a.b.s_off[l]];
  const double tau = f.tk_cnt ? f.tau[l] : 0.0;
  if (f.tk_cnt) {
    const int keep = f.tk_keep[l];
    const int64_t wb = f.tk_wbase[l], tb = f.tk_tbase[l];
    for (int j = lt.tile * blockDim.x + threadIdx.x; j < keep; j += lt.tiles * blockDim.x) f.tk_work[wb + j] = f.tk_top[tb + j];
  }
  // warp-uniform trip count: the threshold keys are appended with one atomic per warp
  for (int i0 = lt.tile * blockDim.x + (threadIdx.x & ~31); i0 < n; i0 += lt.tiles * blockDim.x) {
    const int i = i0 + lane;
    bool pass = false;
    double logp = 0.0;
    const int node = i < n ? f.it_node[base + i] : -1;
    if (i < n && !(i > 0 && f.it_node[base + i - 1] == node)) {
      const int g = f.nd_grp[node];
      double total = neg_inf(), best = neg_inf(), ub = neg_inf();
      int t0 = 0, t1 = 0;
      for (int q = i; q < n && f.it_node[base + q] == node; ++q) {
        const int x = f.it_state[base + q];
        const double cx = a.cont[(long long)x * a.NG + g];
        if (cx > neg_inf()) ub = log_add(ub, f.it_wsum[base + q] + cx);
        const double ex = a.exitw[(long long)x * a.NG + g];
        if (!(ex > neg_inf())) continue;
        total = log_add(total, f.it_wsum[base + q] + ex);
        const double v = f.it_wmax[base + q] + ex;
        const int q0 = f.it_t0[base + q], q1 = a.b.time[x];
        if (v > best || (v == best && (q0 < t0 || (q0 == t0 && q1 < t1)))) {
          best = v;
          t0 = q0;
          t1 = q1;
        }
      }
      f.nd_total[node] = total;
      f.nd_best[node] = best;
      f.nd_t0[node] = t0;
      f.nd_t1[node] = t1;
      f.nd_ub[node] = ub;
      logp = total - beta0;  // as k_char_rowkey forms it
      pass = total > neg_inf() && logp > tau;
    }
    if (f.tk_cnt) {
      const unsigned int m = __ballot_sync(0xffffffffu, pass);
      if (m) {
        const int leader = __ffs(m) - 1;
        int first = 0;
        if (lane == leader) first = atomicAdd(f.tk_cnt + l, __popc(m));
        first = __shfl_sync(0xffffffffu, first, leader);
        if (pass) f.tk_work[f.tk_wbase[l] + first + __popc(m & ((1u << lane) - 1u))] = ~ord_f64(logp + 0.0);
      }
    }
  }
}

// after the sort of the threshold segments (descending log-probability): the nbest best keys
// are carried over to the top buffer, and tau becomes the nbest-th once there are nbest of them
// (unsorted = no segment can hold nbest keys yet: all are carried over, tau stays)
__global__ void __launch_bounds__(256) k_char_tau(Frontier f, const unsigned long long* key_b, const unsigned char* where,
                                                  int sorted, int nbest, unsigned long long* top, int32_t* keep_out,
                                                  double* tau) {
  const int l = blockIdx.x;
  const int n = f.tk_cnt[l];
  const int keep = min(n, nbest);
  const unsigned long long* src = (sorted && where[l] ? key_b : f.tk_work) + f.tk_wbase[l];
  for (int j = threadIdx.x; j < keep; j += blockDim.x) top[f.tk_tbase[l] + j] = src[j];
  __syncthreads();
  if (threadIdx.x == 0) {
    if (sorted && n >= nbest) tau[l] = key_logp(src[nbest - 1]);
    keep_out[l] = keep;
    f.tk_cnt[l] = keep;
  }
}

// expansion: candidates per item = same-group out arcs of its state
__global__ void __launch_bounds__(256) k_char_count(CharArgs a, Frontier f) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const BatchView& b = a.b;
  const int l = lt.l;
  const int n = f.icnt[l];
  const int64_t base = f.ibase[l];
  const double beta0 = a.beta[b.s_off[l]];
  const double tau = f.tau ? f.tau[l] : neg_inf();
  for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
    const int x = f.it_state[base + i];
    const int node = f.it_node[base + i];
    const bool cut = below_cut(f.nd_ub[node] - beta0, tau, beta0);
    if (cut && !f.cut_cnt) {
      f.cand_cnt[base + i] = 0;
      continue;
    }
    const int g = f.nd_grp[node];
    int c = 0;
    for (int k = b.out_off[x]; k < b.out_off[x + 1]; ++k) {
      const int4 r = b.out_rec[k];
      if (group_of(a, r.w) == g && !char_arc_pruned(a, l, x, r.x, r)) ++c;
    }
    if (cut) {  // counted for the debug line only
      if (c) atomicAdd(f.cut_cnt, (unsigned long long)c);
      c = 0;
    }
    f.cand_cnt[base + i] = c;
  }
}

__global__ void __launch_bounds__(256) k_char_expand(CharArgs a, Frontier f) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const BatchView& b = a.b;
  const int l = lt.l;
  const int n = f.icnt[l];
  const int64_t base = f.ibase[l], cb = f.cbase[l];
  for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
    if (f.cand_cnt[base + i] == 0) continue;
    const int x = f.it_state[base + i];
    const int node = f.it_node[base + i];
    const int g = f.nd_grp[node];
    const unsigned long long parent = (unsigned long long)((int64_t)node - f.parent_pool_base - f.ibase[l]);
    int64_t o = cb + f.cand_loc[base + i];
    for (int k = b.out_off[x]; k < b.out_off[x + 1]; ++k) {
      const int4 r = b.out_rec[k];
      if (group_of(a, r.w) != g || char_arc_pruned(a, l, x, r.x, r)) continue;
      const double cost = rec_cost(r, a.cp);
      if (a.segment) {
        f.c_main[o] = (parent << (kKeyCharBits + kKeyStateBits)) | ((unsigned long long)(unsigned int)r.w << kKeyStateBits) |
                      frame_tag(a, r.x, g);
        f.c_state[o] = r.x - b.s_off[l];
        f.ckey[o] = (unsigned long long)(r.x - b.s_off[l]);
      } else {
        f.ckey[o] = (parent << (kKeyCharBits + kKeyStateBits)) | ((unsigned long long)(unsigned int)r.w << kKeyStateBits) |
                    (unsigned long long)(r.x - b.s_off[l]);
      }
      f.cval[o] = (unsigned int)(o - cb);
      f.c_wsum[o] = f.it_wsum[base + i] - cost;
      f.c_wmax[o] = f.it_wmax[base + i] - cost;
      f.c_t0[o] = f.it_t0[base + i];
      ++o;
    }
  }
}

// segment mode, between the two stable sorts: candidates are ordered by destination
// state; give them their main key (always in buffer A) for the second sort
__global__ void __launch_bounds__(256) k_char_rekey(Frontier f, unsigned long long* key_a, unsigned int* val_a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = f.ccnt[l];
  const int64_t cb = f.cbase[l];
  const unsigned int* val = (f.where[l] ? f.val_b : f.val_a) + cb;
  for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
    const unsigned int j = val[i];
    key_a[cb + i] = f.c_main[cb + j];
    val_a[cb + i] = j;
  }
}

// Sorted candidates -> merged items (runs of equal key) and new trie nodes (runs of equal
// (parent, label)); both keep the candidates' slot range.  A lattice's candidates (up to millions
// at the deeper levels) are cut into tiles of 256 handled by many CTAs: COUNT = true leaves the
// item / node heads of every tile in tile_i / tile_n, k_char_tile_scan turns them into the heads
// before the tile, COUNT = false writes the items and nodes.
__device__ __forceinline__ int char_tile_slot(const Frontier& f, int l, int tile) {
  return (int)(f.cbase[l] >> 8) + l + tile;  // disjoint per lattice: ceil(ccnt / 256) <= slots to the next base
}

template <bool COUNT>
__global__ void __launch_bounds__(256) k_char_reduce(CharArgs a, Frontier f) {
  __shared__ int warp_i[8], warp_n[8];
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = f.ccnt[l];
  const int64_t cb = f.cbase[l];
  const unsigned long long* key = (f.where[l] ? f.key_b : f.key_a) + cb;
  const unsigned int* val = (f.where[l] ? f.val_b : f.val_a) + cb;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int tile = lt.tile * 256; tile < n; tile += lt.tiles * 256) {
    const int i = tile + tid;
    unsigned long long k = 0;
    bool ihead = false, nhead = false;
    int st_i = 0;  // lattice-local destination state of candidate i
    if (i < n) {
      k = key[i];
      if (a.segment) {  // key = (parent, label, frame tag); the state rides beside it
        st_i = f.c_state[cb + val[i]];
        nhead = i == 0 || key[i - 1] != k;
        ihead = nhead || f.c_state[cb + val[i - 1]] != st_i;
      } else {
        st_i = (int)(k & ((1ULL << kKeyStateBits) - 1ULL));
        ihead = i == 0 || key[i - 1] != k;
        nhead = i == 0 || (key[i - 1] >> kKeyStateBits) != (k >> kKeyStateBits);
      }
    }
    int xi = ihead ? 1 : 0, xn = nhead ? 1 : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int yi = __shfl_up_sync(0xffffffffu, xi, o), yn = __shfl_up_sync(0xffffffffu, xn, o);
      if (lane >= o) {
        xi += yi;
        xn += yn;
      }
    }
    if (lane == 31) {
      warp_i[warp] = xi;
      warp_n[warp] = xn;
    }
    __syncthreads();
    const int slot_t = char_tile_slot(f, l, tile >> 8);
    if (COUNT) {
      if (tid == 0) {
        int ti = 0, tn = 0;
        for (int w = 0; w < 8; ++w) {
          ti += warp_i[w];
          tn += warp_n[w];
        }
        f.tile_i[slot_t] = ti;
        f.tile_n[slot_t] = tn;
      }
      __syncthreads();
      continue;
    }
    int addi = f.tile_i[slot_t], addn = f.tile_n[slot_t];  // heads of this lattice before the tile
    for (int w = 0; w < warp; ++w) {
      addi += warp_i[w];
      addn += warp_n[w];
    }
    if (ihead) {
      const int slot = addi + xi - 1;       // item rank inside the lattice
      const int nrank = addn + xn - 1;      // node rank inside the lattice (this depth)
      const int64_t node = f.node_pool_base + cb + nrank;
      unsigned int j = val[i];
      double wsum = f.c_wsum[cb + j], wmax = f.c_wmax[cb + j];
      int t0 = f.c_t0[cb + j];
      for (int q = i + 1; q < n && key[q] == k && (!a.segment || f.c_state[cb + val[q]] == st_i); ++q) {
        j = val[q];
        wsum = log_add(wsum, f.c_wsum[cb + j]);
        const double v = f.c_wmax[cb + j];
        const int q0 = f.c_t0[cb + j];
        if (v > wmax || (v == wmax && q0 < t0)) {
          wmax = v;
          t0 = q0;
        }
      }
      f.n_node[cb + slot] = (int32_t)node;
      f.n_state[cb + slot] = a.b.s_off[l] + st_i;
      f.n_wsum[cb + slot] = wsum;
      f.n_wmax[cb + slot] = wmax;
      f.n_t0[cb + slot] = t0;
      if (nhead) {
        const int chr = (int)((k >> kKeyStateBits) & ((1ULL << kKeyCharBits) - 1ULL));
        const long long up = (long long)(k >> (kKeyCharBits + kKeyStateBits));
        f.nd_chr[node] = chr;
        f.nd_lat[node] = l;
        f.nd_total[node] = neg_inf();
        if (f.depth == 0) {
          f.nd_parent[node] = -1;
          f.nd_cnt[node] = (int32_t)up;
          f.nd_grp[node] = group_of(a, chr);
          f.nd_len[node] = 1;
        } else {
          const int64_t parent = f.parent_pool_base + f.ibase[l] + up;
          f.nd_parent[node] = (int32_t)parent;
          f.nd_cnt[node] = f.nd_cnt[parent];
          f.nd_grp[node] = f.nd_grp[parent];
          f.nd_len[node] = f.nd_len[parent] + 1;
        }
      }
    }
    __syncthreads();  // warp_i / warp_n are rewritten by the next tile
  }
}

// one CTA per lattice: exclusive scan of its tiles' head counts; the lattice's item count
__global__ void __launch_bounds__(256) k_char_tile_scan(Frontier f) {
  __shared__ int warp_i[8], warp_n[8];
  __shared__ int carry_i, carry_n;
  const int l = blockIdx.x;
  const int nt = (f.ccnt[l] + 255) >> 8;
  const int s0 = char_tile_slot(f, l, 0);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_i = carry_n = 0;
  __syncthreads();
  for (int base = 0; base < nt; base += 256) {
    const int t = base + tid;
    const int ci = t < nt ? f.tile_i[s0 + t] : 0, cn = t < nt ? f.tile_n[s0 + t] : 0;
    int xi = ci, xn = cn;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int yi = __shfl_up_sync(0xffffffffu, xi, o), yn = __shfl_up_sync(0xffffffffu, xn, o);
      if (lane >= o) {
        xi += yi;
        xn += yn;
      }
    }
    if (lane == 31) {
      warp_i[warp] = xi;
      warp_n[warp] = xn;
    }
    __syncthreads();
    int addi = carry_i, addn = carry_n;
    for (int w = 0; w < warp; ++w) {
      addi += warp_i[w];
      addn += warp_n[w];
    }
    if (t < nt) {
      f.tile_i[s0 + t] = addi + xi - ci;
      f.tile_n[s0 + t] = addn + xn - cn;
    }
    __syncthreads();
    if (tid == 255) {
      carry_i = addi + xi;
      carry_n = addn + xn;
    }
    __syncthreads();
  }
  if (tid == 0) f.ncnt[l] = carry_i;
}

// ---- 4b. lattice-char-index-utterance: exact occurrence probabilities ---------------------------
// For a pseudo-word v (group gv, |v| = m) a first-occurrence DP over the split lattice (SURVEY.md
// App. B.2 for characters), cells per state x:
//   a0[x][g]   (g < NG) paths start -> x whose last arc has group g, that are not inside a run matching
//              a prefix of v and have completed no occurrence of v;
//   a[x][j]    (j = 1..m) the same inside a run of group gv whose labels so far spell v[0..j).
// An arc x -> y of label c and group gy != g_x starts a run (to a[y][1] if gy = gv and c = v[0], else
// to a0[y][gy]); when it leaves a[x][m] it completes an occurrence instead.  A same-group arc goes from
// a[x][j] to a[x][j+1] if c = v[j], else to a0 (a run longer than v, or another string).  Completions
// at x are the exit mass: P(v) = log-sum over x of a[x][m] + exit[x][gv].  Costs and beam tests are
// those of the frontier.  Below the level where v's first character can be entered (the earliest state
// of v's depth-0 ancestor) a0 = A and a = -inf; after the level of v's last item no completion is
// possible: the DP runs over that level span only, a warp per node, its cells in a scratch chunk.
//   PHASE 0: per item slot the scratch a node's DP needs (0 = no DP), the roots' first states, and the
//            carried-over threshold keys (k_char_accum gathers none in this mode);
//   PHASE 1: the DP of every slot with scratch, over the slots of a chunk of lattices; its value
//            becomes the node's row value and goes to the threshold segment;
//   PHASE 2: after the last depth, row values below the lattice's final tau are dropped (the rows
//            left are the nbest best and whatever ties the nbest-th; the host breaks those ties).
struct OccArgs {
  double* nd_occ;              // per node: log-sum of the occurrence paths (row value), -inf = none
  int32_t* nd_lo;              // per depth-0 node: its first item state
  int32_t* need;               // per item slot: scratch doubles of its node's DP
  const int32_t* loc;          // lattice-local exclusive scan of need
  const int64_t* sbase;        // [L+1] first scratch double of each lattice
  double* scratch;
  int64_t chunk_base;          // scratch holds [chunk_base, chunk_base + capacity) of the batch
  int64_t slot0, slot1;        // PHASE 1: item slots of the chunk
  int64_t pool;                // PHASE 2: node pool slots in use
  const int32_t* nd_lat;
  unsigned long long* tasks;   // KLU_CHAR_DEBUG: DP tasks of this depth (else nullptr)
};

__device__ __forceinline__ int state_level(const CharArgs& a, int l, int s) {
  const int* lv = a.b.lvl_start + a.b.lvl_off[l];
  return last_le(lv, 0, a.b.lvl_off[l + 1] - a.b.lvl_off[l] - 1, s);
}

// level span [*j0, *j1] of node's DP (items [i, ...) of the current depth, first of the node)
__device__ __forceinline__ void occ_span(const CharArgs& a, const Frontier& f, const OccArgs& q, int l, int64_t base,
                                         int n, int i, int node, int* j0, int* j1) {
  int root = node;
  while (f.nd_parent[root] >= 0) root = f.nd_parent[root];
  int k = i;
  while (k + 1 < n && f.it_node[base + k + 1] == node) ++k;  // items are sorted by state: the last one is the latest
  *j0 = state_level(a, l, q.nd_lo[root]);
  *j1 = state_level(a, l, f.it_state[base + k]);
}

__device__ __forceinline__ double occ_a0(const CharArgs& a, int l, const double* sc, int s_lo, int W, int x, int g) {
  if (x >= s_lo) return sc[(long long)(x - s_lo) * W + g];
  if (a.nhi[x] < a.nlo[x]) return neg_inf();
  return a.A[cell_of(a, l, x) + g];
}

template <int PHASE>
__global__ void __launch_bounds__(256) k_char_occ(CharArgs a, Frontier f, OccArgs q) {
  if (PHASE == 2) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < q.pool; i += (int64_t)gridDim.x * blockDim.x) {
      const int l = q.nd_lat[i];
      if (l < 0 || !(q.nd_occ[i] > neg_inf())) continue;
      if (!(q.nd_occ[i] - a.beta[a.b.s_off[l]] >= f.tau[l])) q.nd_occ[i] = neg_inf();
    }
    return;
  }
  const int NG = a.NG;
  if (PHASE == 0) {
    const LatTile lt = lat_tile();
    const int l = lt.l;
    const int n = f.icnt[l];
    const int64_t base = f.ibase[l];
    const double beta0 = a.beta[a.b.s_off[l]];
    const double tau = f.tau[l];
    if (f.tk_cnt) {
      const int keep = f.tk_keep[l];
      const int64_t wb = f.tk_wbase[l], tb = f.tk_tbase[l];
      for (int j = lt.tile * blockDim.x + threadIdx.x; j < keep; j += lt.tiles * blockDim.x) f.tk_work[wb + j] = f.tk_top[tb + j];
    }
    for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
      const int node = f.it_node[base + i];
      int need = 0;
      if (!(i > 0 && f.it_node[base + i - 1] == node)) {
        q.nd_occ[node] = neg_inf();
        if (f.depth == 0) q.nd_lo[node] = f.it_state[base + i];
        const double total = f.nd_total[node];
        if (total > neg_inf() && !below_cut(total - beta0, tau, beta0)) {
          int j0, j1;
          occ_span(a, f, q, l, base, n, i, node, &j0, &j1);
          const int* lv = a.b.lvl_start + a.b.lvl_off[l];
          const int m = f.nd_len[node];
          need = (lv[j1 + 1] - lv[j0]) * (NG + m) + (m + 1) / 2;
          if (q.tasks) atomicAdd(q.tasks, 1ULL);
        }
      }
      q.need[base + i] = need;
    }
    return;
  }
  // PHASE 1: a warp per task; the warps of the grid take 32 slots at a time
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const BatchView& b = a.b;
  for (int64_t s32 = q.slot0 + gw * 32; s32 < q.slot1; s32 += nwarps * 32) {
    const int64_t s = s32 + lane;
    unsigned int todo = __ballot_sync(0xffffffffu, s < q.slot1 && q.need[s] > 0);
    while (todo) {
      const int64_t slot = s32 + __ffs(todo) - 1;
      todo &= todo - 1;
      const int l = last_le(f.ibase, 0, b.L - 1, slot);
      const int64_t base = f.ibase[l];
      const int i = (int)(slot - base), n = f.icnt[l];
      if (i >= n) continue;  // a slot past the lattice's items (PHASE 0 left its need unwritten)
      const int node = f.it_node[slot];
      const int g = f.nd_grp[node], m = f.nd_len[node], W = NG + m;
      int j0, j1;
      occ_span(a, f, q, l, base, n, i, node, &j0, &j1);
      const int* lv = b.lvl_start + b.lvl_off[l];
      const int s_lo = lv[j0];
      double* sc = q.scratch + (q.sbase[l] + q.loc[slot] - q.chunk_base);
      int* v = reinterpret_cast<int*>(sc + (long long)(lv[j1 + 1] - s_lo) * W);
      if (lane == 0) {
        int p = m, x = node;
        while (x >= 0) {
          v[--p] = f.nd_chr[x];
          x = f.nd_parent[x];
        }
      }
      __syncwarp();
      double res = neg_inf();
      for (int j = j0; j <= j1; ++j) {
        const int y0 = lv[j], ny = lv[j + 1] - y0;
        for (int c = lane; c < ny * W; c += 32) {
          const int y = y0 + c / W, k = c % W;
          double acc = neg_inf();
          for (int e = b.in_off[y]; e < b.in_off[y + 1]; ++e) {
            const int4 r = b.in_rec[e];
            const int ge = group_of(a, r.w);
            if (k < NG ? ge != k : (ge != g || r.w != v[k - NG])) continue;
            const int x = r.x;
            if (char_arc_pruned(a, l, x, y, r)) continue;
            const double cost = rec_cost(r, a.cp);
            if (k < NG) {
              const bool first = k == g && r.w == v[0];  // a new run here matches v[0]
              for (int gu = 0; gu < NG; ++gu) {
                if (first && gu != k) continue;
                const double xv = occ_a0(a, l, sc, s_lo, W, x, gu);
                if (xv > neg_inf()) acc = log_add(acc, xv - cost);
              }
              if (x >= s_lo)
                for (int jj = 1; jj <= m; ++jj) {
                  if (k != g ? jj == m : (jj < m && r.w == v[jj])) continue;  // completed / matched on
                  const double xv = sc[(long long)(x - s_lo) * W + NG + jj - 1];
                  if (xv > neg_inf()) acc = log_add(acc, xv - cost);
                }
            } else if (k == NG) {  // a[y][1]: a run entered with v[0]
              for (int gu = 0; gu < NG; ++gu) {
                if (gu == g) continue;
                const double xv = occ_a0(a, l, sc, s_lo, W, x, gu);
                if (xv > neg_inf()) acc = log_add(acc, xv - cost);
              }
            } else if (x >= s_lo) {  // a[y][j], j >= 2
              const double xv = sc[(long long)(x - s_lo) * W + k - 1];
              if (xv > neg_inf()) acc = log_add(acc, xv - cost);
            }
          }
          sc[(long long)(y - s_lo) * W + k] = acc;
          if (k == W - 1 && acc > neg_inf()) {
            const double ex = a.exitw[(long long)y * NG + g];
            if (ex > neg_inf()) res = log_add(res, acc + ex);
          }
        }
        __syncwarp();
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) res = log_add(res, __shfl_xor_sync(0xffffffffu, res, o));
      if (lane == 0) {
        q.nd_occ[node] = res;
        const double logp = res - a.beta[b.s_off[l]];  // as k_char_rowkey forms it
        if (f.tk_cnt && res > neg_inf() && logp > f.tau[l])
          f.tk_work[f.tk_wbase[l] + atomicAdd(f.tk_cnt + l, 1)] = ~ord_f64(logp + 0.0);
      }
      __syncwarp();
    }
  }
}

// ---- 5. rows -----------------------------------------------------------------------
struct RowArgs {
  int64_t pool;             // nodes in the pool
  const int32_t *nd_lat, *nd_parent, *nd_chr, *nd_cnt, *nd_t0, *nd_t1, *nd_len;
  const double* nd_total;
  const double* beta;
  const int32_t* s_off;
  int32_t* row_cnt;         // [L]
  const int64_t* row_base;  // [L]
  int32_t* cursor;          // [L]
  unsigned long long* key;
  unsigned int* val;
  const unsigned long long *key_a, *key_b;
  const unsigned int *val_a, *val_b;
  const unsigned char* where;
  int nbest;
  // selected rows
  const int64_t* out_base;  // [L+1]
  int32_t *o_node, *o_pos, *o_t0, *o_t1, *o_len;
  double* o_logp;
  const int64_t* chr_off;   // per selected row
  int32_t* o_chars;
};

// (pool slots of one lattice are contiguous per depth, so a warp's rows nearly always belong to one
// lattice: the lanes are grouped by lattice and one atomic per group is issued)
__global__ void __launch_bounds__(256) k_char_rowcount(RowArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const int64_t rounds = (a.pool + stride - 1) / stride;
  for (int64_t r = 0; r < rounds; ++r) {
    const int64_t i = r * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int l = -1;
    if (i < a.pool) {
      l = a.nd_lat[i];
      if (l >= 0 && !(a.nd_total[i] > neg_inf())) l = -1;
    }
    const unsigned int grp = __match_any_sync(0xffffffffu, l);
    if (l >= 0 && lane == __ffs(grp) - 1) atomicAdd(a.row_cnt + l, __popc(grp));
  }
}

// rows into per-lattice segments (arrival order; the two stable sorts that follow make it deterministic)
__global__ void __launch_bounds__(256) k_char_rowfill(RowArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const int64_t rounds = (a.pool + stride - 1) / stride;
  for (int64_t r = 0; r < rounds; ++r) {
    const int64_t i = r * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int l = -1;
    if (i < a.pool) {
      l = a.nd_lat[i];
      if (l >= 0 && !(a.nd_total[i] > neg_inf())) l = -1;
    }
    const unsigned int grp = __match_any_sync(0xffffffffu, l);
    const int leader = __ffs(grp) - 1;
    int first = 0;
    if (l >= 0 && lane == leader) first = atomicAdd(a.cursor + l, __popc(grp));
    first = __shfl_sync(0xffffffffu, first, leader);
    if (l < 0) continue;
    const int64_t o = a.row_base[l] + first + __popc(grp & ((1u << lane) - 1u));
    a.key[o] = (unsigned long long)i;  // first sort: node id (creation order = depth, then key order)
    a.val[o] = (unsigned int)i;
  }
}

// second sort key: descending log-probability
__global__ void __launch_bounds__(256) k_char_rowkey(RowArgs a, int L) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = a.row_cnt[l];
  const int64_t base = a.row_base[l];
  const unsigned int* val = (a.where[l] ? a.val_b : a.val_a) + base;
  for (int i = lt.tile * blockDim.x + threadIdx.x; i < n; i += lt.tiles * blockDim.x) {
    const unsigned int node = val[i];
    const double logp = a.nd_total[node] - a.beta[a.s_off[l]];
    a.key[base + i] = ~ord_f64(logp + 0.0);
    a.val[base + i] = node;
  }
}

__global__ void __launch_bounds__(256) k_char_select(RowArgs a) {
  const int l = blockIdx.x;
  const int n = min(a.row_cnt[l], a.nbest);
  const int64_t base = a.row_base[l], ob = a.out_base[l];
  const unsigned int* val = (a.where[l] ? a.val_b : a.val_a) + base;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < n; i += gridDim.y * blockDim.x) {
    const int node = (int)val[i];
    a.o_node[ob + i] = node;
    a.o_pos[ob + i] = a.nd_cnt[node];
    a.o_t0[ob + i] = a.nd_t0[node];
    a.o_t1[ob + i] = a.nd_t1[node];
    a.o_len[ob + i] = a.nd_len[node];
    a.o_logp[ob + i] = a.nd_total[node] - a.beta[a.s_off[l]];
  }
}

__global__ void __launch_bounds__(256) k_char_chars(RowArgs a, int64_t rows) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += stride) {
    int node = a.o_node[i];
    int64_t p = a.chr_off[i + 1];
    while (node >= 0) {
      a.o_chars[--p] = a.nd_chr[node];
      node = a.nd_parent[node];
    }
  }
}

// grows a device buffer, keeping its first `keep` bytes
int grow_keep(klu_ctx* c, DevBuf& b, size_t keep, size_t need) {
  if (need <= b.cap) return 0;
  DevBuf nb;
  KLU_TRY(nb.reserve(std::max(need, b.cap * 2)));
  if (keep) KLU_CUDA(cudaMemcpyAsync(nb.p, b.p, keep, cudaMemcpyDeviceToDevice, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  b.release();
  b = nb;
  return 0;
}

struct CharState {
  std::vector<int64_t> row_off;  // [L+1] selected rows per lattice
  std::vector<int64_t> chr_off;  // per selected row (+1)
  std::vector<int32_t> chars, pos, t0, t1;
  std::vector<double> logp;
};

CharState& char_state(klu_ctx* c) {
  if (!c->char_state) c->char_state = new CharState();
  return *static_cast<CharState*>(c->char_state);
}

}  // namespace

// segment: lattice-char-index-segment keys (frame tags); utterance: lattice-char-index-utterance
// (string keys, rows valued by k_char_occ); neither: lattice-char-index-position
int run_char_index(klu_ctx* c, const klu_opts* o, bool segment, bool utterance) {
  const int32_t L = c->L;
  for (int32_t l = 0; l < L; ++l)
    if (!c->h_times_ok[l]) {
      set_error("lattice " + std::to_string(l) + ": inconsistent state times (lattice is not aligned)");
      return 1;
    }
  const bool use_beam = o->beam != INFINITY;
  if (use_beam && !(o->beam > 0.0f)) {
    set_error("--beam must be positive");
    return 1;
  }
  if (o->nbest < 0) {
    set_error("--nbest must not be negative");
    return 1;
  }
  CostParams cp = make_cost_params(o, false);
  if (use_beam) KLU_TRY(run_tropical_sweeps(c, cp));
  KLU_TRY(run_log_sweeps(c, cp, use_beam, o->beam));
  CharState& out = char_state(c);
  out = CharState();
  out.row_off.assign(L + 1, 0);
  out.chr_off.assign(1, 0);
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = 0;
  c->last_chars = 0;
  if (L == 0 || c->S == 0) return 0;
  if (c->max_states >= (1 << kKeyStateBits) || c->max_label >= (1 << kKeyCharBits) ||
      (segment && c->max_time + 1 >= (1 << kKeyStateBits))) {
    set_error("char index: more than 2^20 states (or frames) per lattice or labels above 2^20 are not supported");
    return 1;
  }
  // ---- dense label groups (kwsbin2/utils.h:41-84) ----
  std::vector<int32_t> gids;
  for (int32_t i = 0; i < o->num_group_labels; ++i) gids.push_back(o->group_ids[i]);
  for (int32_t i = 0; i < o->num_inc_groups; ++i) gids.push_back(o->inc_groups[i]);
  for (int32_t i = 0; i < o->num_del_groups; ++i) gids.push_back(o->del_groups[i]);
  gids.push_back(0);
  gids.push_back(INT_MAX);
  std::sort(gids.begin(), gids.end());
  gids.erase(std::unique(gids.begin(), gids.end()), gids.end());
  if (gids.size() > 32) {
    set_error("char index: more than 32 label groups");
    return 1;
  }
  auto dense = [&](int32_t g) { return (int)(std::lower_bound(gids.begin(), gids.end(), g) - gids.begin()); };
  std::vector<std::pair<int32_t, int32_t> > lg;
  for (int32_t i = 0; i < o->num_group_labels; ++i) lg.push_back(std::make_pair(o->group_labels[i], dense(o->group_ids[i])));
  lg.push_back(std::make_pair(0, dense(0)));  // epsilon is its own group
  std::sort(lg.begin(), lg.end());
  lg.erase(std::unique(lg.begin(), lg.end(), [](const std::pair<int32_t, int32_t>& x, const std::pair<int32_t, int32_t>& y) {
             return x.first == y.first;
           }),
           lg.end());
  std::vector<int32_t> glabels, gdense;
  for (auto& kv : lg) {
    glabels.push_back(kv.first);
    gdense.push_back(kv.second);
  }
  const size_t S = (size_t)c->S, E = (size_t)std::max<int64_t>(c->E, 1);
  enum { C_GL = 0, C_GD, C_NLO, C_NHI, C_CCNT, C_CLOC, C_CBASE, C_A, C_EXIT, C_TOT, C_CONT };
  DevBuf* sc = c->d_scratch;
  KLU_TRY(sc[C_GL].reserve(4 * glabels.size()));
  KLU_TRY(sc[C_GD].reserve(4 * glabels.size()));
  KLU_CUDA(cudaMemcpyAsync(sc[C_GL].p, glabels.data(), 4 * glabels.size(), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemcpyAsync(sc[C_GD].p, gdense.data(), 4 * gdense.size(), cudaMemcpyHostToDevice, c->stream));
  KLU_TRY(sc[C_NLO].reserve(4 * S));
  KLU_TRY(sc[C_NHI].reserve(4 * S));
  KLU_TRY(sc[C_CCNT].reserve(4 * S));
  KLU_TRY(sc[C_CLOC].reserve(4 * S));
  KLU_TRY(sc[C_CBASE].reserve(8 * (size_t)(L + 1)));
  KLU_TRY(sc[C_TOT].reserve(8 * (size_t)(L + 1)));
  CharArgs a;
  memset(&a, 0, sizeof(a));
  a.b = c->view();
  a.cp = cp;
  a.glabels = sc[C_GL].as<int32_t>();
  a.gdense = sc[C_GD].as<int32_t>();
  a.ngl = (int)glabels.size();
  a.NG = (int)gids.size();
  a.dflt = dense(INT_MAX);
  a.eps = dense(0);
  a.segment = segment ? 1 : 0;
  // the segment tool has no word-count split (kwsbin2/lattice-char-index-segment.cc:113-117), nor has
  // the utterance tool (its keys are the strings alone)
  for (int32_t i = 0; !segment && !utterance && i < o->num_inc_groups; ++i) a.inc_mask |= 1u << dense(o->inc_groups[i]);
  for (int32_t i = 0; i < o->num_del_groups; ++i) a.del_mask |= 1u << dense(o->del_groups[i]);
  a.use_beam = use_beam ? 1 : 0;
  a.vfwd = c->d_vfwd.as<double>();
  a.vbwd = c->d_vbwd.as<double>();
  a.best = c->d_best.as<double>();
  a.beam = (double)o->beam;
  a.beta = c->d_beta.as<double>();
  a.nlo = sc[C_NLO].as<int32_t>();
  a.nhi = sc[C_NHI].as<int32_t>();
  a.cell_cnt = sc[C_CCNT].as<int32_t>();
  a.cell_loc = sc[C_CLOC].as<int32_t>();
  a.cell_base = sc[C_CBASE].as<int64_t>();
  const int lat_warps_grid = (L * 32 + 127) / 128;
  int64_t max_arcs = 0;
  for (int32_t l = 0; l < L; ++l) max_arcs = std::max(max_arcs, c->h_e_off[l + 1] - c->h_e_off[l]);
  const int arc_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  const int st_tiles = (int)std::max<int64_t>(1, std::min<int64_t>(((int64_t)c->max_states * a.NG + 255) / 256, 64));
  {
    KLU_LAUNCH(c, "k_char_bands");
    k_char_bands<<<lat_warps_grid, 128, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_char_bands"));
  // per-lattice scans go through this helper: counts -> local offsets (device), totals -> bases (host)
  std::vector<long long> h_tot(L);
  std::vector<int64_t> h_base(L + 1);
  auto scan = [&](const SegRange& rg, const int32_t* cnt, int32_t* loc, int64_t* d_base) -> int {
    {
      KLU_LAUNCH(c, "k_char_scan");
      k_char_scan<<<L, 256, 0, c->stream>>>(rg, cnt, loc, sc[C_TOT].as<long long>());
    }
    KLU_TRY(check_launch("k_char_scan"));
    KLU_CUDA(cudaMemcpyAsync(h_tot.data(), sc[C_TOT].p, 8 * (size_t)L, cudaMemcpyDeviceToHost, c->stream));
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    h_base[0] = 0;
    for (int32_t l = 0; l < L; ++l) {
      if (h_tot[l] >= ((long long)1 << 31)) {
        set_error("char index: more than 2^31 work items in lattice " + std::to_string(l));
        return 1;
      }
      h_base[l + 1] = h_base[l] + h_tot[l];
    }
    KLU_CUDA(cudaMemcpyAsync(d_base, h_base.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  };
  SegRange states_rg = {a.b.s_off, nullptr, nullptr};
  KLU_TRY(scan(states_rg, a.cell_cnt, sc[C_CLOC].as<int32_t>(), sc[C_CBASE].as<int64_t>()));
  const int64_t cells = h_base[L];
  KLU_TRY(sc[C_A].reserve(8 * (size_t)std::max<int64_t>(cells, 1)));
  KLU_TRY(sc[C_EXIT].reserve(8 * S * (size_t)a.NG));
  a.A = sc[C_A].as<double>();
  a.exitw = sc[C_EXIT].as<double>();
  {
    KLU_LAUNCH(c, "k_char_fwd");
    k_char_fwd<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_char_fwd"));
  {
    KLU_LAUNCH(c, "k_char_exit");
    k_char_exit<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_char_exit"));
  KLU_TRY(sc[C_CONT].reserve(8 * S * (size_t)a.NG));
  a.cont = sc[C_CONT].as<double>();
  {
    KLU_LAUNCH(c, "k_char_cont");
    k_char_cont<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_char_cont"));

  // ---- frontier buffers (grown as needed) ----
  // The frontier, trie and row buffers live in the context (c->d_char) and are reused from run to
  // run: allocating and freeing ~50 buffers per run cost more than the kernels on small batches.
  int nbuf = 0;
  auto buf = [&]() -> DevBuf& { return c->d_char[nbuf++]; };
  DevBuf &it_node = buf(), &it_state = buf(), &it_t0 = buf(), &it_wsum = buf(), &it_wmax = buf();  // current items
  DevBuf &n_node = buf(), &n_state = buf(), &n_t0 = buf(), &n_wsum = buf(), &n_wmax = buf();       // next items
  DevBuf &ckey_a = buf(), &ckey_b = buf(), &cval_a = buf(), &cval_b = buf(), &c_wsum = buf(), &c_wmax = buf(),
         &c_t0 = buf(), &c_state = buf(), &c_main = buf(), &cand_cnt = buf(), &cand_loc = buf(), &where = buf();
  DevBuf &nd_parent = buf(), &nd_chr = buf(), &nd_cnt = buf(), &nd_grp = buf(), &nd_lat = buf(), &nd_t0 = buf(),
         &nd_t1 = buf(), &nd_len = buf(), &nd_total = buf(), &nd_best = buf(), &nd_ub = buf();
  DevBuf &d_ibase = buf(), &d_icnt = buf(), &d_cbase = buf(), &d_ccnt = buf(), &d_ncnt = buf();
  DevBuf &tile_i = buf(), &tile_n = buf();
  // n-best cut: per-lattice threshold segments (work keys + sort buffers), carried-over keys (top),
  // [L] counts / tau, [3 (L+1)] bases (work, top of the last depth, top of this depth), debug count
  DevBuf &tk_work = buf(), &tk_keyb = buf(), &tk_vala = buf(), &tk_valb = buf(), &tk_top = buf(), &tk_where = buf(),
         &tk_cnt = buf(), &tk_keep = buf(), &tk_tau = buf(), &tk_bases = buf(), &d_cut = buf();
  KLU_TRY(d_ibase.reserve(8 * (size_t)(L + 1)));
  KLU_TRY(d_icnt.reserve(4 * (size_t)L));
  KLU_TRY(d_cbase.reserve(8 * (size_t)(L + 1)));
  KLU_TRY(d_ccnt.reserve(4 * (size_t)L));
  KLU_TRY(d_ncnt.reserve(4 * (size_t)L));
  KLU_TRY(where.reserve((size_t)L));
  KLU_TRY(cand_cnt.reserve(4 * E));
  KLU_TRY(cand_loc.reserve(4 * E));
  int64_t pool = 0;  // node pool slots in use
  // utterance: per node its row value and (depth 0) first state; per item slot the DP scratch it
  // needs, its scan, the lattices' scratch bases, the scratch, the debug task count
  DevBuf &nd_occ = buf(), &nd_lo = buf(), &occ_need = buf(), &occ_loc = buf(), &occ_base = buf(), &occ_scratch = buf(),
         &d_tasks = buf();
  DevBuf* nd_all[13] = {&nd_parent, &nd_chr, &nd_cnt, &nd_grp, &nd_lat, &nd_t0, &nd_t1, &nd_len, &nd_total, &nd_best, &nd_ub,
                        &nd_occ, &nd_lo};
  auto grow_pool = [&](int64_t need) -> int {
    for (int i = 0; i < (utterance ? 13 : 11); ++i) {
      const size_t w = (i >= 8 && i <= 11) ? 8 : 4;
      KLU_TRY(grow_keep(c, *nd_all[i], (size_t)pool * w, (size_t)need * w));
    }
    return 0;
  };
  Frontier f;
  memset(&f, 0, sizeof(f));
  int64_t items_total = 0;            // slots of the current item arrays
  std::vector<int32_t> h_cnt(L);
  int64_t parent_pool_base = 0;
  // n-best cut state: tau starts at -inf (+inf with nbest 0: no row is selected, nothing is
  // expanded); a lattice's threshold keys are gathered from depth 1 on
  const int nbest = o->nbest;
  const bool debug = getenv("KLU_CHAR_DEBUG") != nullptr;
  std::vector<int64_t> h_seen(L, 0);  // items folded so far per lattice (>= its final nodes)
  std::vector<int64_t> h_tkb(3 * (size_t)(L + 1), 0);  // work | top of the last depth | top of this depth
  KLU_TRY(tk_cnt.reserve(4 * (size_t)L));
  KLU_TRY(tk_keep.reserve(4 * (size_t)L));
  KLU_TRY(tk_tau.reserve(8 * (size_t)L));
  KLU_TRY(tk_where.reserve((size_t)L));
  KLU_TRY(tk_bases.reserve(8 * h_tkb.size()));
  KLU_TRY(d_cut.reserve(8));
  {
    const std::vector<double> tau0(L, nbest > 0 ? -INFINITY : INFINITY);
    KLU_CUDA(cudaMemcpyAsync(tk_tau.p, tau0.data(), 8 * (size_t)L, cudaMemcpyHostToDevice, c->stream));
    KLU_CUDA(cudaMemsetAsync(tk_cnt.p, 0, 4 * (size_t)L, c->stream));
    KLU_CUDA(cudaMemsetAsync(tk_keep.p, 0, 4 * (size_t)L, c->stream));
    KLU_CUDA(cudaStreamSynchronize(c->stream));  // tau0 leaves scope
  }
  f.tau = tk_tau.as<double>();
  f.tk_keep = tk_keep.as<int32_t>();
  f.tk_wbase = tk_bases.as<int64_t>();
  f.tk_tbase = tk_bases.as<int64_t>() + (L + 1);
  unsigned long long h_cut = 0;
  // threshold step of one depth: lay out the segments (carried-over keys + this depth's items per
  // lattice), let k_char_accum fill them, sort, carry the nbest best over and update tau
  auto cut_layout = [&]() -> int {
    int64_t w = 0, t = 0;
    for (int32_t l = 0; l <= L; ++l) h_tkb[(size_t)(L + 1) + l] = h_tkb[2 * (size_t)(L + 1) + l];  // top of the last depth
    const int64_t t_last = h_tkb[2 * (size_t)(L + 1) - 1];
    for (int32_t l = 0; l < L; ++l) {
      h_tkb[l] = w;
      w += std::min<int64_t>(nbest, h_seen[l]) + h_cnt[l];
      h_seen[l] += h_cnt[l];
      h_tkb[2 * (size_t)(L + 1) + l] = t;
      t += std::min<int64_t>(nbest, h_seen[l]);
    }
    h_tkb[L] = w;
    h_tkb[2 * (size_t)(L + 1) + L] = t;
    KLU_TRY(tk_work.reserve(8 * (size_t)std::max<int64_t>(w, 1)));
    KLU_TRY(tk_keyb.reserve(8 * (size_t)std::max<int64_t>(w, 1)));
    KLU_TRY(tk_vala.reserve(4 * (size_t)std::max<int64_t>(w, 1)));
    KLU_TRY(tk_valb.reserve(4 * (size_t)std::max<int64_t>(w, 1)));
    // the top buffer keeps the last depth's keys until k_char_accum has copied them
    KLU_TRY(grow_keep(c, tk_top, 8 * (size_t)t_last, 8 * (size_t)std::max<int64_t>(std::max(t, t_last), 1)));
    KLU_CUDA(cudaMemcpyAsync(tk_bases.p, h_tkb.data(), 8 * h_tkb.size(), cudaMemcpyHostToDevice, c->stream));
    f.tk_work = tk_work.as<unsigned long long>();
    f.tk_top = tk_top.as<unsigned long long>();
    f.tk_tbase = tk_bases.as<int64_t>() + (L + 1);
    return 0;
  };
  auto cut_update = [&]() -> int {
    bool full = false;  // some lattice may hold nbest keys: sort
    for (int32_t l = 0; l < L; ++l) full = full || h_seen[l] >= nbest;
    SegSortArgs ss;
    ss.seg_base = tk_bases.as<int64_t>();
    ss.seg_cnt = tk_cnt.as<int32_t>();
    ss.key_a = tk_work.as<unsigned long long>();
    ss.val_a = tk_vala.as<unsigned int>();
    ss.key_b = tk_keyb.as<unsigned long long>();
    ss.val_b = tk_valb.as<unsigned int>();
    ss.where = tk_where.as<unsigned char>();
    ss.lo_bit = 0;
    ss.hi_bit = 64;
    if (full) {
      {
        KLU_LAUNCH(c, "k_seg_radix_sort");
        KLU_TRY(seg_sort_launch(c, ss, L, h_tkb[L]));
      }
      KLU_TRY(check_launch("k_seg_radix_sort(char cut)"));
    }
    Frontier g = f;
    g.tk_tbase = tk_bases.as<int64_t>() + 2 * (L + 1);  // this depth's top layout
    {
      KLU_LAUNCH(c, "k_char_tau");
      k_char_tau<<<L, 256, 0, c->stream>>>(g, ss.key_b, ss.where, full ? 1 : 0, nbest, tk_top.as<unsigned long long>(),
                                           tk_keep.as<int32_t>(), tk_tau.as<double>());
    }
    KLU_TRY(check_launch("k_char_tau"));
    return 0;
  };
  // utterance: the occurrence DPs of the nodes just folded (k_char_occ), in chunks of lattices whose
  // scratch fits kOccChunk doubles
  std::vector<int64_t> h_ibase(L + 1, 0);  // item slots of the current depth per lattice
  OccArgs q;
  memset(&q, 0, sizeof(q));
  auto occ_depth = [&](int node_depth) -> int {
    q.nd_occ = nd_occ.as<double>();
    q.nd_lo = nd_lo.as<int32_t>();
    KLU_TRY(occ_need.reserve(4 * (size_t)std::max<int64_t>(items_total, 1)));
    KLU_TRY(occ_loc.reserve(4 * (size_t)std::max<int64_t>(items_total, 1)));
    KLU_TRY(occ_base.reserve(8 * (size_t)(L + 1)));
    q.need = occ_need.as<int32_t>();
    q.loc = occ_loc.as<int32_t>();
    q.sbase = occ_base.as<int64_t>();
    q.tasks = nullptr;
    if (debug) {
      KLU_TRY(d_tasks.reserve(8));
      KLU_CUDA(cudaMemsetAsync(d_tasks.p, 0, 8, c->stream));
      q.tasks = d_tasks.as<unsigned long long>();
    }
    {
      KLU_LAUNCH(c, "k_char_occ");
      k_char_occ<0><<<dim3(L, 64), 256, 0, c->stream>>>(a, f, q);
    }
    KLU_TRY(check_launch("k_char_occ(count)"));
    SegRange rg = {nullptr, f.ibase, f.icnt};
    KLU_TRY(scan(rg, q.need, occ_loc.as<int32_t>(), occ_base.as<int64_t>()));
    const std::vector<int64_t> sb = h_base;  // scratch doubles before each lattice
    if (debug) {
      unsigned long long h_tasks = 0;
      KLU_CUDA(cudaMemcpyAsync(&h_tasks, d_tasks.p, 8, cudaMemcpyDeviceToHost, c->stream));
      KLU_CUDA(cudaStreamSynchronize(c->stream));
      fprintf(stderr, "[klu char] depth %d: %llu occurrence DP tasks, %lld scratch doubles\n", node_depth, h_tasks,
              (long long)sb[L]);
    }
    q.tasks = nullptr;
    constexpr int64_t kOccChunk = (int64_t)1 << 27;  // 1 GiB of scratch
    for (int32_t l0 = 0; l0 < L;) {
      int32_t l1 = l0 + 1;
      while (l1 < L && sb[l1 + 1] - sb[l0] <= kOccChunk) ++l1;
      const int64_t need = sb[l1] - sb[l0];
      if (need > 0) {
        KLU_TRY(occ_scratch.reserve(8 * (size_t)need));
        q.scratch = occ_scratch.as<double>();
        q.chunk_base = sb[l0];
        q.slot0 = h_ibase[l0];
        q.slot1 = h_ibase[l1];
        const int64_t warps = std::max<int64_t>(1, (q.slot1 - q.slot0 + 31) / 32);
        {
          KLU_LAUNCH(c, "k_char_occ");
          k_char_occ<1><<<(unsigned)std::min<int64_t>((warps + 7) / 8, (int64_t)c->num_sms * 8), 256, 0, c->stream>>>(a, f, q);
        }
        KLU_TRY(check_launch("k_char_occ"));
      }
      l0 = l1;
    }
    return 0;
  };
  for (int depth = 0; depth < 100000; ++depth) {
    // ---- candidates: count, scan ----
    if (depth == 0) {
      f.cand_cnt = cand_cnt.as<int32_t>();
      f.cand_loc = cand_loc.as<int32_t>();
      {
        KLU_LAUNCH(c, "k_char_count0");
        k_char_count0<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a, f);
      }
      KLU_TRY(check_launch("k_char_count0"));
      SegRange rg = {a.b.e_off, nullptr, nullptr};
      KLU_TRY(scan(rg, f.cand_cnt, cand_loc.as<int32_t>(), d_cbase.as<int64_t>()));
    } else {
      KLU_TRY(cand_cnt.reserve(4 * (size_t)std::max<int64_t>(items_total, 1)));
      KLU_TRY(cand_loc.reserve(4 * (size_t)std::max<int64_t>(items_total, 1)));
      f.cand_cnt = cand_cnt.as<int32_t>();
      f.cand_loc = cand_loc.as<int32_t>();
      if (nbest > 0) {
        KLU_TRY(cut_layout());
        f.tk_cnt = tk_cnt.as<int32_t>();
      }
      {
        Frontier g = f;
        if (utterance) g.tk_cnt = nullptr;  // the threshold keys are the occurrence values (k_char_occ)
        KLU_LAUNCH(c, "k_char_accum");
        k_char_accum<<<dim3(L, 64), 256, 0, c->stream>>>(a, g);
      }
      KLU_TRY(check_launch("k_char_accum"));
      if (utterance) KLU_TRY(occ_depth(depth - 1));
      if (nbest > 0) KLU_TRY(cut_update());
      if (debug) {
        KLU_CUDA(cudaMemsetAsync(d_cut.p, 0, 8, c->stream));
        f.cut_cnt = d_cut.as<unsigned long long>();
      }
      {
        KLU_LAUNCH(c, "k_char_count");
        k_char_count<<<dim3(L, 64), 256, 0, c->stream>>>(a, f);
      }
      KLU_TRY(check_launch("k_char_count"));
      SegRange rg = {nullptr, f.ibase, f.icnt};
      KLU_TRY(scan(rg, f.cand_cnt, cand_loc.as<int32_t>(), d_cbase.as<int64_t>()));
    }
    const int64_t ncand = h_base[L];
    if (debug) {
      long long mx = 0;
      for (int32_t l = 0; l < L; ++l) mx = std::max(mx, h_tot[l]);
      if (depth > 0) {
        KLU_CUDA(cudaMemcpyAsync(&h_cut, d_cut.p, 8, cudaMemcpyDeviceToHost, c->stream));
        KLU_CUDA(cudaStreamSynchronize(c->stream));
      }
      fprintf(stderr, "[klu char] depth %d: %lld candidates (largest lattice %lld), %llu cut, pool %lld, items %lld\n",
              depth, (long long)ncand, mx, depth > 0 ? h_cut : 0ULL, (long long)pool, (long long)items_total);
    }
    if (ncand == 0) break;
    for (int32_t l = 0; l < L; ++l) {
      h_cnt[l] = (int32_t)h_tot[l];
      if (h_tot[l] >= ((long long)1 << kKeyParentBits)) {
        set_error("char index: more than 2^24 trie nodes at one depth in lattice " + std::to_string(l));
        return 1;
      }
    }
    KLU_CUDA(cudaMemcpyAsync(d_ccnt.p, h_cnt.data(), 4 * (size_t)L, cudaMemcpyHostToDevice, c->stream));
    KLU_TRY(ckey_a.reserve(8 * (size_t)ncand));
    KLU_TRY(ckey_b.reserve(8 * (size_t)ncand));
    KLU_TRY(cval_a.reserve(4 * (size_t)ncand));
    KLU_TRY(cval_b.reserve(4 * (size_t)ncand));
    KLU_TRY(c_wsum.reserve(8 * (size_t)ncand));
    KLU_TRY(c_wmax.reserve(8 * (size_t)ncand));
    KLU_TRY(c_t0.reserve(4 * (size_t)ncand));
    if (segment) {
      KLU_TRY(c_state.reserve(4 * (size_t)ncand));
      KLU_TRY(c_main.reserve(8 * (size_t)ncand));
    }
    KLU_TRY(n_node.reserve(4 * (size_t)ncand));
    KLU_TRY(n_state.reserve(4 * (size_t)ncand));
    KLU_TRY(n_t0.reserve(4 * (size_t)ncand));
    KLU_TRY(n_wsum.reserve(8 * (size_t)ncand));
    KLU_TRY(n_wmax.reserve(8 * (size_t)ncand));
    if (pool + ncand >= ((int64_t)1 << 31)) {
      set_error("char index: more than 2^31 trie nodes in one batch; split it");
      return 1;
    }
    KLU_TRY(grow_pool(pool + ncand));
    KLU_CUDA(cudaMemsetAsync(nd_lat.as<int32_t>() + pool, 0xff, 4 * (size_t)ncand, c->stream));  // unused slots: lattice -1
    f.nd_parent = nd_parent.as<int32_t>();
    f.nd_chr = nd_chr.as<int32_t>();
    f.nd_cnt = nd_cnt.as<int32_t>();
    f.nd_grp = nd_grp.as<int32_t>();
    f.nd_lat = nd_lat.as<int32_t>();
    f.nd_t0 = nd_t0.as<int32_t>();
    f.nd_t1 = nd_t1.as<int32_t>();
    f.nd_len = nd_len.as<int32_t>();
    f.nd_total = nd_total.as<double>();
    f.nd_best = nd_best.as<double>();
    f.nd_ub = nd_ub.as<double>();
    f.cbase = d_cbase.as<int64_t>();
    f.ccnt = d_ccnt.as<int32_t>();
    f.ckey = ckey_a.as<unsigned long long>();
    f.cval = cval_a.as<unsigned int>();
    f.c_wsum = c_wsum.as<double>();
    f.c_wmax = c_wmax.as<double>();
    f.c_t0 = c_t0.as<int32_t>();
    f.c_state = c_state.as<int32_t>();
    f.c_main = c_main.as<unsigned long long>();
    f.depth = depth;
    f.parent_pool_base = parent_pool_base;
    f.node_pool_base = pool;
    if (depth == 0) {
      KLU_LAUNCH(c, "k_char_emit0");
      k_char_emit0<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a, f);
    } else {
      KLU_LAUNCH(c, "k_char_expand");
      k_char_expand<<<dim3(L, 64), 256, 0, c->stream>>>(a, f);
    }
    KLU_TRY(check_launch("k_char_expand"));
    SegSortArgs ss;
    ss.seg_base = d_cbase.as<int64_t>();
    ss.seg_cnt = d_ccnt.as<int32_t>();
    ss.key_a = ckey_a.as<unsigned long long>();
    ss.val_a = cval_a.as<unsigned int>();
    ss.key_b = ckey_b.as<unsigned long long>();
    ss.val_b = cval_b.as<unsigned int>();
    ss.where = where.as<unsigned char>();
    ss.lo_bit = 0;
    ss.hi_bit = segment ? kKeyStateBits : 64;  // segment mode: by destination state first ...
    {
      KLU_LAUNCH(c, "k_seg_radix_sort");
      KLU_TRY(seg_sort_launch(c, ss, L, ncand));
    }
    KLU_TRY(check_launch("k_seg_radix_sort(char)"));
    if (segment) {  // ... then, stably, by (parent, label, frame tag)
      f.key_a = ss.key_a;
      f.key_b = ss.key_b;
      f.val_a = ss.val_a;
      f.val_b = ss.val_b;
      f.where = ss.where;
      int64_t max_c = 0;
      for (int32_t l = 0; l < L; ++l) max_c = std::max<int64_t>(max_c, h_cnt[l]);
      {
        KLU_LAUNCH(c, "k_char_rekey");
        k_char_rekey<<<dim3(L, (unsigned)std::max<int64_t>(1, std::min<int64_t>((max_c + 255) / 256, 64))), 256, 0,
                       c->stream>>>(f, ss.key_a, ss.val_a);
      }
      KLU_TRY(check_launch("k_char_rekey"));
      ss.hi_bit = 64;
      {
        KLU_LAUNCH(c, "k_seg_radix_sort");
        KLU_TRY(seg_sort_launch(c, ss, L, ncand));
      }
      KLU_TRY(check_launch("k_seg_radix_sort(char keys)"));
    }
    f.key_a = ss.key_a;
    f.key_b = ss.key_b;
    f.val_a = ss.val_a;
    f.val_b = ss.val_b;
    f.where = ss.where;
    f.n_node = n_node.as<int32_t>();
    f.n_state = n_state.as<int32_t>();
    f.n_t0 = n_t0.as<int32_t>();
    f.n_wsum = n_wsum.as<double>();
    f.n_wmax = n_wmax.as<double>();
    f.ncnt = d_ncnt.as<int32_t>();
    {
      int64_t max_c = 0;
      for (int32_t l = 0; l < L; ++l) max_c = std::max<int64_t>(max_c, h_cnt[l]);
      const size_t slots = (size_t)(ncand >> 8) + (size_t)L + 2;
      KLU_TRY(tile_i.reserve(4 * slots));
      KLU_TRY(tile_n.reserve(4 * slots));
      f.tile_i = tile_i.as<int32_t>();
      f.tile_n = tile_n.as<int32_t>();
      const unsigned rt = (unsigned)std::max<int64_t>(1, std::min<int64_t>((max_c + 255) / 256, 2048));
      {
        KLU_LAUNCH(c, "k_char_reduce");
        k_char_reduce<true><<<dim3(L, rt), 256, 0, c->stream>>>(a, f);
      }
      KLU_TRY(check_launch("k_char_reduce(count)"));
      {
        KLU_LAUNCH(c, "k_char_tile_scan");
        k_char_tile_scan<<<L, 256, 0, c->stream>>>(f);
      }
      KLU_TRY(check_launch("k_char_tile_scan"));
      {
        KLU_LAUNCH(c, "k_char_reduce");
        k_char_reduce<false><<<dim3(L, rt), 256, 0, c->stream>>>(a, f);
      }
    }
    KLU_TRY(check_launch("k_char_reduce"));
    // ---- the merged items become the current frontier (they keep the candidates' slot ranges) ----
    std::swap(it_node, n_node);
    std::swap(it_state, n_state);
    std::swap(it_t0, n_t0);
    std::swap(it_wsum, n_wsum);
    std::swap(it_wmax, n_wmax);
    std::swap(d_ibase, d_cbase);
    std::swap(d_icnt, d_ncnt);
    f.ibase = d_ibase.as<int64_t>();
    f.icnt = d_icnt.as<int32_t>();
    f.it_node = it_node.as<int32_t>();
    f.it_state = it_state.as<int32_t>();
    f.it_t0 = it_t0.as<int32_t>();
    f.it_wsum = it_wsum.as<double>();
    f.it_wmax = it_wmax.as<double>();
    items_total = ncand;
    parent_pool_base = pool;
    pool += ncand;
    if (utterance) h_ibase = h_base;
  }
  if (pool == 0) return 0;
  if (utterance && nbest > 0) {  // rows: the nbest best occurrence values and their ties
    q.pool = pool;
    q.nd_lat = nd_lat.as<int32_t>();
    q.nd_occ = nd_occ.as<double>();
    {
      KLU_LAUNCH(c, "k_char_occ");
      k_char_occ<2><<<(unsigned)std::max<int64_t>(1, std::min<int64_t>((pool + 255) / 256, (int64_t)c->num_sms * 8)), 256, 0,
                      c->stream>>>(a, f, q);
    }
    KLU_TRY(check_launch("k_char_occ(rows)"));
  }
  // ---- rows ----
  DevBuf &row_cnt = buf(), &row_base = buf(), &cursor = buf(), &rkey_a = buf(), &rkey_b = buf(), &rval_a = buf(),
         &rval_b = buf(), &out_base = buf(), &o_node = buf(), &chr_off = buf();
  KLU_TRY(row_cnt.reserve(4 * (size_t)L));
  KLU_TRY(cursor.reserve(4 * (size_t)L));
  KLU_TRY(row_base.reserve(8 * (size_t)(L + 1)));
  KLU_TRY(out_base.reserve(8 * (size_t)(L + 1)));
  KLU_CUDA(cudaMemsetAsync(row_cnt.p, 0, 4 * (size_t)L, c->stream));
  KLU_CUDA(cudaMemsetAsync(cursor.p, 0, 4 * (size_t)L, c->stream));
  RowArgs r;
  memset(&r, 0, sizeof(r));
  r.pool = pool;
  r.nd_lat = nd_lat.as<int32_t>();
  r.nd_parent = nd_parent.as<int32_t>();
  r.nd_chr = nd_chr.as<int32_t>();
  r.nd_cnt = nd_cnt.as<int32_t>();
  r.nd_t0 = nd_t0.as<int32_t>();
  r.nd_t1 = nd_t1.as<int32_t>();
  r.nd_len = nd_len.as<int32_t>();
  r.nd_total = utterance ? nd_occ.as<double>() : nd_total.as<double>();
  r.beta = a.beta;
  r.s_off = a.b.s_off;
  r.row_cnt = row_cnt.as<int32_t>();
  r.cursor = cursor.as<int32_t>();
  r.nbest = utterance ? INT_MAX : o->nbest;  // utterance: ties at the cut are broken on the host
  {
    KLU_LAUNCH(c, "k_char_rowcount");
    k_char_rowcount<<<c->num_sms * 4, 256, 0, c->stream>>>(r);
  }
  KLU_TRY(check_launch("k_char_rowcount"));
  std::vector<int32_t> h_rows(L);
  KLU_CUDA(cudaMemcpyAsync(h_rows.data(), row_cnt.p, 4 * (size_t)L, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  std::vector<int64_t> h_rbase(L + 1, 0), h_obase(L + 1, 0);
  for (int32_t l = 0; l < L; ++l) {
    h_rbase[l + 1] = h_rbase[l] + h_rows[l];
    h_obase[l + 1] = h_obase[l] + std::min<int64_t>(h_rows[l], r.nbest);
  }
  const int64_t nrows = h_rbase[L], nsel = h_obase[L];
  out.row_off = h_obase;
  c->h_res_off = h_obase;
  c->last_entries = nsel;
  if (nsel == 0) return 0;
  KLU_CUDA(cudaMemcpyAsync(row_base.p, h_rbase.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemcpyAsync(out_base.p, h_obase.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_TRY(rkey_a.reserve(8 * (size_t)nrows));
  KLU_TRY(rkey_b.reserve(8 * (size_t)nrows));
  KLU_TRY(rval_a.reserve(4 * (size_t)nrows));
  KLU_TRY(rval_b.reserve(4 * (size_t)nrows));
  r.row_base = row_base.as<int64_t>();
  r.key = rkey_a.as<unsigned long long>();
  r.val = rval_a.as<unsigned int>();
  {
    KLU_LAUNCH(c, "k_char_rowfill");
    k_char_rowfill<<<c->num_sms * 4, 256, 0, c->stream>>>(r);
  }
  KLU_TRY(check_launch("k_char_rowfill"));
  SegSortArgs ss;
  ss.seg_base = row_base.as<int64_t>();
  ss.seg_cnt = row_cnt.as<int32_t>();
  ss.key_a = rkey_a.as<unsigned long long>();
  ss.val_a = rval_a.as<unsigned int>();
  ss.key_b = rkey_b.as<unsigned long long>();
  ss.val_b = rval_b.as<unsigned int>();
  ss.where = where.as<unsigned char>();
  ss.lo_bit = 0;
  ss.hi_bit = 32;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, ss, L, nrows));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(rows by node)"));
  int64_t max_rows = 0;
  for (int32_t l = 0; l < L; ++l) max_rows = std::max<int64_t>(max_rows, h_rows[l]);
  const int row_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_rows + 255) / 256, 64));
  r.key_a = ss.key_a;
  r.key_b = ss.key_b;
  r.val_a = ss.val_a;
  r.val_b = ss.val_b;
  r.where = ss.where;
  // the keyed copy goes to a fresh pair of buffers so that a lattice whose first sort
  // ended in either buffer is read consistently
  DevBuf &k2a = buf(), &k2b = buf(), &v2a = buf(), &v2b = buf(), &where2 = buf();
  KLU_TRY(k2a.reserve(8 * (size_t)nrows));
  KLU_TRY(k2b.reserve(8 * (size_t)nrows));
  KLU_TRY(v2a.reserve(4 * (size_t)nrows));
  KLU_TRY(v2b.reserve(4 * (size_t)nrows));
  KLU_TRY(where2.reserve((size_t)L));
  r.key = k2a.as<unsigned long long>();
  r.val = v2a.as<unsigned int>();
  {
    KLU_LAUNCH(c, "k_char_rowkey");
    k_char_rowkey<<<dim3(L, row_tiles), 256, 0, c->stream>>>(r, L);
  }
  KLU_TRY(check_launch("k_char_rowkey"));
  ss.key_a = k2a.as<unsigned long long>();
  ss.val_a = v2a.as<unsigned int>();
  ss.key_b = k2b.as<unsigned long long>();
  ss.val_b = v2b.as<unsigned int>();
  ss.where = where2.as<unsigned char>();
  ss.hi_bit = 64;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, ss, L, nrows));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(rows by logp)"));
  r.key_a = ss.key_a;
  r.key_b = ss.key_b;
  r.val_a = ss.val_a;
  r.val_b = ss.val_b;
  r.where = ss.where;
  // selected rows -> d_res columns
  KLU_TRY(o_node.reserve(4 * (size_t)nsel));
  KLU_TRY(c->d_res[0].reserve(4 * (size_t)nsel));  // length
  KLU_TRY(c->d_res[1].reserve(4 * (size_t)nsel));  // pos
  KLU_TRY(c->d_res[2].reserve(4 * (size_t)nsel));  // t0
  KLU_TRY(c->d_res[3].reserve(4 * (size_t)nsel));  // t1
  KLU_TRY(c->d_res[4].reserve(8 * (size_t)nsel));  // logp
  r.out_base = out_base.as<int64_t>();
  r.o_node = o_node.as<int32_t>();
  r.o_len = c->d_res[0].as<int32_t>();
  r.o_pos = c->d_res[1].as<int32_t>();
  r.o_t0 = c->d_res[2].as<int32_t>();
  r.o_t1 = c->d_res[3].as<int32_t>();
  r.o_logp = c->d_res[4].as<double>();
  {
    KLU_LAUNCH(c, "k_char_select");
    k_char_select<<<dim3(L, std::max(1, std::min((o->nbest + 255) / 256, 64))), 256, 0, c->stream>>>(r);
  }
  KLU_TRY(check_launch("k_char_select"));
  std::vector<int32_t> h_len(nsel);
  out.pos.resize(nsel);
  out.t0.resize(nsel);
  out.t1.resize(nsel);
  out.logp.resize(nsel);
  KLU_CUDA(cudaMemcpyAsync(h_len.data(), c->d_res[0].p, 4 * (size_t)nsel, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaMemcpyAsync(out.pos.data(), c->d_res[1].p, 4 * (size_t)nsel, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaMemcpyAsync(out.t0.data(), c->d_res[2].p, 4 * (size_t)nsel, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaMemcpyAsync(out.t1.data(), c->d_res[3].p, 4 * (size_t)nsel, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaMemcpyAsync(out.logp.data(), c->d_res[4].p, 8 * (size_t)nsel, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  out.chr_off.assign(nsel + 1, 0);
  for (int64_t i = 0; i < nsel; ++i) out.chr_off[i + 1] = out.chr_off[i] + h_len[i];
  const int64_t nchars = out.chr_off[nsel];
  KLU_TRY(chr_off.reserve(8 * (size_t)(nsel + 1)));
  KLU_TRY(c->d_res[6].reserve(4 * (size_t)std::max<int64_t>(nchars, 1)));
  KLU_CUDA(cudaMemcpyAsync(chr_off.p, out.chr_off.data(), 8 * (size_t)(nsel + 1), cudaMemcpyHostToDevice, c->stream));
  r.chr_off = chr_off.as<int64_t>();
  r.o_chars = c->d_res[6].as<int32_t>();
  {
    KLU_LAUNCH(c, "k_char_chars");
    k_char_chars<<<std::max<int64_t>(1, std::min<int64_t>((nsel + 255) / 256, c->num_sms * 8)), 256, 0, c->stream>>>(r, nsel);
  }
  KLU_TRY(check_launch("k_char_chars"));
  out.chars.resize(nchars);
  KLU_CUDA(cudaMemcpyAsync(out.chars.data(), c->d_res[6].p, 4 * (size_t)nchars, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  // ---- final order of each lattice's rows (kwsbin2/lattice-char-index-position.cc:272-281):
  //      logp desc, string asc (decimal labels joined by '_', compared as text), position asc;
  //      the utterance tool keeps the first nbest of that order (a tie at the cut goes to the
  //      smaller string: its rows are the nbest best and everything tied with the nbest-th)
  {
    std::vector<std::string> str(nsel);
    for (int64_t i = 0; i < nsel; ++i) {
      std::string& s = str[i];
      for (int64_t k = out.chr_off[i]; k < out.chr_off[i + 1]; ++k) {
        if (k > out.chr_off[i]) s += "_";
        s += std::to_string(out.chars[k]);
      }
    }
    std::vector<int64_t> perm(nsel);
    for (int64_t i = 0; i < nsel; ++i) perm[i] = i;
    for (int32_t l = 0; l < L; ++l)
      std::sort(perm.begin() + h_obase[l], perm.begin() + h_obase[l + 1], [&](int64_t x, int64_t y) {
        if (out.logp[x] != out.logp[y]) return out.logp[x] > out.logp[y];
        if (str[x] != str[y]) return str[x] < str[y];
        if (!segment) return out.pos[x] < out.pos[y];
        // kwsbin2/lattice-char-index-segment.cc:205-219: then initial frame, then final frame
        if (out.t0[x] != out.t0[y]) return out.t0[x] < out.t0[y];
        return out.t1[x] < out.t1[y];
      });
    CharState s2;
    s2.row_off.assign(L + 1, 0);
    s2.chr_off.assign(1, 0);
    for (int32_t l = 0; l < L; ++l) {
      const int64_t end = std::min<int64_t>(h_obase[l + 1], h_obase[l] + std::max(o->nbest, 0));  // (utterance: the cut)
      for (int64_t i = h_obase[l]; i < end; ++i) {
        const int64_t p = perm[i];
        s2.pos.push_back(out.pos[p]);
        s2.t0.push_back(out.t0[p]);
        s2.t1.push_back(out.t1[p]);
        s2.logp.push_back(out.logp[p]);
        s2.chars.insert(s2.chars.end(), out.chars.begin() + out.chr_off[p], out.chars.begin() + out.chr_off[p + 1]);
        s2.chr_off.push_back((int64_t)s2.chars.size());
      }
      s2.row_off[l + 1] = (int64_t)s2.pos.size();
    }
    out = s2;
  }
  c->h_res_off = out.row_off;
  c->last_entries = out.row_off[L];
  c->last_chars = (int64_t)out.chars.size();
  return 0;
}

int run_char_position(klu_ctx* c, const klu_opts* o) { return run_char_index(c, o, false, false); }
int run_char_segment(klu_ctx* c, const klu_opts* o) { return run_char_index(c, o, true, false); }
int run_char_utterance(klu_ctx* c, const klu_opts* o) { return run_char_index(c, o, false, true); }

void char_release(klu_ctx* c) {
  delete static_cast<CharState*>(c->char_state);
  c->char_state = nullptr;
  for (DevBuf& b : c->d_char) b.release();
}

}  // namespace klu

using namespace klu;

extern "C" {

int klu_result_char_sizes(klu_ctx* c, int64_t* total_chars) {
  if (c->last_tool != KLU_CHAR_POSITION && c->last_tool != KLU_CHAR_SEGMENT && c->last_tool != KLU_CHAR_UTTERANCE) {
    set_error("klu_result_char_sizes: last run was not a char index tool");
    return 1;
  }
  *total_chars = c->last_chars;
  return 0;
}

int klu_fetch_char_position(klu_ctx* c, int64_t* char_off, int32_t* chars, int32_t* pos, int32_t* t0, int32_t* t1,
                            double* logp) {
  if (c->last_tool != KLU_CHAR_POSITION) {
    set_error("klu_fetch_char_position: last run was not KLU_CHAR_POSITION");
    return 1;
  }
  if (!c->char_state) {
    set_error("klu_fetch_char_position: no results");
    return 1;
  }
  const CharState& s = *static_cast<const CharState*>(c->char_state);
  const size_t n = s.pos.size();
  if (char_off) memcpy(char_off, s.chr_off.data(), 8 * (n + 1));
  if (chars && !s.chars.empty()) memcpy(chars, s.chars.data(), 4 * s.chars.size());
  if (pos && n) memcpy(pos, s.pos.data(), 4 * n);
  if (t0 && n) memcpy(t0, s.t0.data(), 4 * n);
  if (t1 && n) memcpy(t1, s.t1.data(), 4 * n);
  if (logp && n) memcpy(logp, s.logp.data(), 8 * n);
  return 0;
}

int klu_fetch_char_segment(klu_ctx* c, int64_t* char_off, int32_t* chars, int32_t* t0, int32_t* t1, double* logp) {
  if (c->last_tool != KLU_CHAR_SEGMENT) {
    set_error("klu_fetch_char_segment: last run was not KLU_CHAR_SEGMENT");
    return 1;
  }
  c->last_tool = KLU_CHAR_POSITION;  // same row store
  const int rc = klu_fetch_char_position(c, char_off, chars, nullptr, t0, t1, logp);
  c->last_tool = KLU_CHAR_SEGMENT;
  return rc;
}

int klu_fetch_char_utterance(klu_ctx* c, int64_t* char_off, int32_t* chars, double* logp) {
  if (c->last_tool != KLU_CHAR_UTTERANCE) {
    set_error("klu_fetch_char_utterance: last run was not KLU_CHAR_UTTERANCE");
    return 1;
  }
  c->last_tool = KLU_CHAR_POSITION;  // same row store
  const int rc = klu_fetch_char_position(c, char_off, chars, nullptr, nullptr, nullptr, logp);
  c->last_tool = KLU_CHAR_UTTERANCE;
  return rc;
}

}  // extern "C"
