// klu_sweep.cu -- level-synchronous semiring sweeps (SURVEY.md K2, K3, K5, K9).
//
//   log semiring   ComputeLatticeAlphasAndBetas [ext] (called at
//                  kwsbin2/lattice-word-index-position.cc:66, -segment.cc:63,
//                  latbin/lattice-to-word-frame-post.cc:89, lattice-best-path2.cc:118)
//                  and ComputeCompactLatticeBetas [ext] (-utterance.cc:121-123)
//   tropical       the Viterbi forward/backward of PruneLattice [ext] and
//                  ComputeLatticeBeam (latbin/lattice-prune-dyn-beam.cc:27-90)
//   banded log     alpha over (state, #labels so far): the forward half of the
//                  lattice that DisambiguateStateInputSequenceLength
//                  (fstext/fstext-utils2.h:109-215) would materialise.
//
// Log sweeps: a warp takes 32/G lattices of one direction from a queue sorted by
// descending arc count, and a tile of G lanes sweeps one of them level by level
// (log_sweep_tiles).  A tile stages a batch of a level's arc records in shared
// memory, forms every arc's exp term around one shared reference point, and adds
// each state's terms with a few lanes.  State scores are written to global memory
// and to a per-tile shared-memory ring of recent states; the far end of an arc is
// read from the ring when it is still there, else gathered from global memory.
#include <stdlib.h>

#include "klu_common.cuh"

namespace klu {

namespace {

struct SweepArgs {
  BatchView b;
  CostParams cp;
  double* alpha;
  double* beta;
  const double* vfwd;  // tropical scores for inline --beam pruning (or null)
  const double* vbwd;
  const double* best;  // per lattice best final cost
  double beam;         // (double)(float)beam
  int* counter;
  int do_fwd, do_bwd;
};

// PruneLattice's arc test, evaluated on the fly: the arc is dropped when
// fwd[s] + (cost + bwd[next]) > best_final + beam.
__device__ __forceinline__ bool arc_pruned(const SweepArgs& a, int l, int src, int dst, const int4& r) {
  CostParams cp = a.cp;
  cp.float_sum = 0;  // PruneLattice always uses ConvertToCost (double sum)
  const double cost = rec_cost(r, cp);
  const double fb = __dadd_rn(a.vfwd[src], __dadd_rn(cost, a.vbwd[dst]));
  return fb > __dadd_rn(a.best[l], a.beam);
}
__device__ __forceinline__ bool final_pruned(const SweepArgs& a, int l, int s, double) {
  CostParams cp = a.cp;
  cp.float_sum = 0;
  const double fcost = final_cost(a.b.fin_g[s], a.b.fin_a[s], cp);
  return __dadd_rn(fcost, a.vfwd[s]) > __dadd_rn(a.best[l], a.beam) && fcost != pos_inf();
}

// most recent state scores of a tile kept in shared memory (a ring indexed by state id)
__host__ __device__ constexpr int sweep_ring(int G) { return G >= 8 ? 128 : 32; }
constexpr int kSweepCapPerLane = 8;  // arcs staged per batch = 8 x (lanes of the tile), 16 bytes each

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const unsigned int sa = (unsigned int)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  const unsigned int sa = (unsigned int)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

template <bool FWD, bool BEAM>
__device__ __forceinline__ bool sweep_arc_pruned(const SweepArgs& a, int l, int e, const int4& r) {
  // FWD walks in-order arcs (r.x = source), BWD out-order arcs (r.x = destination)
  const int src = FWD ? r.x : a.b.out_src[e];
  const int dst = FWD ? a.b.out_rec[a.b.in2out[e]].x : r.x;
  return arc_pruned(a, l, src, dst, r);
}

// Exact log-sum of ONE state by ONE lane: max first, then max + log1p(sum of the
// other terms) with libm's exp and log1p (for two terms exactly Kaldi's LogAdd).
// Used for states with more arcs than a tile stages and whenever the fast path's
// shared reference point would under- or overflow.
template <bool FWD, bool BEAM>
__device__ __noinline__ double sweep_state_exact(const SweepArgs& a, int l, int s) {
  const BatchView& b = a.b;
  const int4* rec = FWD ? b.in_rec : b.out_rec;
  const int* off = FWD ? b.in_off : b.out_off;
  const double* score = FWD ? a.alpha : a.beta;
  const int e0 = off[s], e1 = off[s + 1];
  double fin = neg_inf();
  if (!FWD) {
    const double fc = final_cost(b.fin_g[s], b.fin_a[s], a.cp);
    if (!(BEAM && final_pruned(a, l, s, fc))) fin = -fc;
  }
  double m = fin;
  int arg = fin > neg_inf() ? -2 : -1;  // -2: the final weight is the max
  for (int e = e0; e < e1; ++e) {
    const int4 r = __ldg(rec + e);
    if (BEAM && sweep_arc_pruned<FWD, BEAM>(a, l, e, r)) continue;
    const double x = score[r.x] - rec_cost(r, a.cp);
    if (x > m) {
      m = x;
      arg = e;
    }
  }
  if (!(m > neg_inf())) return neg_inf();
  double sum = 0.0;
  if (fin > neg_inf() && arg != -2) sum = exp(fin - m);
  for (int e = e0; e < e1; ++e) {
    if (e == arg) continue;
    const int4 r = __ldg(rec + e);
    if (BEAM && sweep_arc_pruned<FWD, BEAM>(a, l, e, r)) continue;
    sum += exp(score[r.x] - rec_cost(r, a.cp) - m);
  }
  return m + log1p(sum);
}

// Level-synchronous sweep of 32 / G (lattice, direction) items by one warp: a tile
// of G lanes owns one lattice, and the 32 / G tiles run in lockstep so that every
// issued instruction works for all of them (the level loop of a lattice is a long
// dependent chain; what the machine can overlap is OTHER lattices).
//
// Inside a level a tile cuts the states into batches of <= G states and
// <= kCap = 8 G arcs.  The arcs of a batch are one contiguous run of 16-byte records
// (in_rec is sorted by destination, out_rec by source): the tile's lanes stream
// them, each lane turns its arcs into exp(score[other] - cost - ref) and parks the
// term in shared memory.  `ref` is the score of the previous batch's first state: a
// point on the frontier, within a few tens of every term, so one shared reference
// replaces the per-state max of the textbook log-sum-exp (no second pass over the
// arcs).  A few lanes per state then add the state's terms in arc order and
// score = ref + log(sum).  States with one or two terms use Kaldi's LogAdd form
// exactly; sums that leave [1e-280, 1e280] (reference point too far, unreachable
// states, ...) are redone exactly.
template <int G, bool FWD, bool BEAM>
__device__ void log_sweep_tiles(const SweepArgs& a, int first, int lane, double2* xwarp, double* rwarp) {
  constexpr int kCap = kSweepCapPerLane * G;
  constexpr int kRing = sweep_ring(G);
  constexpr int kLog2G = G == 32 ? 5 : G == 16 ? 4 : G == 8 ? 3 : G == 4 ? 2 : 1;
  const BatchView& b = a.b;
  const int gi = lane / G, sl = lane % G;
  const unsigned int gmask = (G == 32 ? 0xffffffffu : ((1u << G) - 1u)) << (gi * G);
  double2* xbuf = xwarp + gi * kCap;  // per arc: the record, then {cost, score}, then {exp term, -}
  double* ring = rwarp + gi * kRing;
  const int4* rec = FWD ? b.in_rec : b.out_rec;
  const int* off = FWD ? b.in_off : b.out_off;
  double* score = FWD ? a.alpha : a.beta;
  bool done = first + gi >= b.L;
  const int l = done ? 0 : b.order[first + gi];
  const int s_begin = b.s_off[l];
  if (!done && s_begin == b.s_off[l + 1]) done = true;
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  double ref = 0.0;
  int j = FWD ? 1 : nl - 1;
  if (FWD && !done)
    for (int s = lv[0] + sl; s < lv[1]; s += G) {
      const double v = (s == s_begin) ? 0.0 : neg_inf();
      score[s] = v;
      ring[s & (kRing - 1)] = v;
    }
  if (!done && (FWD ? j >= nl : j < 0)) done = true;
  int a0 = 0, a1 = 0, s0 = 0;
  int wide = 0x7fffffff;  // backward: first state of the nearest level above the current one wider than kRing
  if (!done) {
    s0 = a0 = lv[j];
    a1 = lv[j + 1];
  }
  __syncwarp();
  while (!__all_sync(0xffffffffu, done)) {
    // ---- the next batch of this tile's current level
    const int idx = s0 + sl;
    int o_lo = 0, o_hi = 0;
    if (!done) {
      o_lo = off[min(idx, a1)];
      o_hi = off[min(idx + 1, a1)];
    }
    const int base = __shfl_sync(0xffffffffu, o_lo, 0, G);
    const unsigned int fit = __ballot_sync(0xffffffffu, !done && idx < a1 && o_hi - base <= kCap) & gmask;
    const int c = __popc(fit);  // states of the batch: the longest prefix whose arcs fit the staging buffer
    const int o_last = __shfl_sync(0xffffffffu, o_hi, max(c - 1, 0), G);
    const int nb = c > 0 ? o_last - base : 0;
    if (!done && c > 0) {  // pull the records a few levels ahead into L2
      const int pf = base + nb + kCap + sl * 8;
      if (sl * 8 < nb && pf < b.E) asm volatile("prefetch.global.L2 [%0];" ::"l"(rec + pf));
    }
    // Passes over the lane's own arcs, each a batch of independent memory operations:
    // (1) the 16-byte records, global -> shared, asynchronously; (2) cost from the record
    // and the other end's score -- from the tile's shared-memory ring of recent scores
    // when it is still there, else gathered asynchronously into the slot -- and the exp
    // term; (3) the exp terms of the gathered ones.
    // Ring slot t & (kRing - 1) still holds state t while no state t +- m kRing was written
    // after it.  Forward, states are written in ascending order, so every t >= a1 - kRing
    // is intact.  Backward, levels go down but the states of a level go up: t < a0 + kRing
    // keeps the current level's writes off t's slot, and t < wide keeps t out of levels
    // wider than kRing, where t + kRing of t's own level was written after t.
    for (int i = sl; i < nb; i += G) cp_async16(xbuf + i, rec + base + i);
    cp_async_wait_all();
    unsigned int pending = 0;
    {
      int it = 0;
      for (int i = sl; i < nb; i += G, ++it) {
        const int4 r = *reinterpret_cast<const int4*>(xbuf + i);
        double cost = rec_cost(r, a.cp);
        if (BEAM && sweep_arc_pruned<FWD, BEAM>(a, l, base + i, r)) cost = pos_inf();
        const int t = r.x;
        if (FWD ? (t >= a1 - kRing) : (t < min(a0 + kRing, wide))) {
          xbuf[i].x = fast_exp(ring[t & (kRing - 1)] - cost - ref);
        } else {
          xbuf[i].x = cost;
          cp_async8(&xbuf[i].y, score + t);
          pending |= 1u << it;
        }
      }
    }
    if (__any_sync(0xffffffffu, pending != 0)) {
      cp_async_wait_all();
      int it = 0;
      for (int i = sl; i < nb; i += G, ++it) {
        if ((pending >> it) & 1u) {
          const double2 v = xbuf[i];
          xbuf[i].x = fast_exp(v.y - v.x - ref);
        }
      }
    }
    __syncwarp();
    // ---- G / pow2ceil(c) lanes per state add its terms, then fold across those lanes
    const int sh = c <= 1 ? kLog2G : kLog2G - (32 - __clz(c - 1));  // log2(lanes per state)
    const int gp = 1 << sh;
    const int st = sl >> sh, sub = sl & (gp - 1);
    const int lo = __shfl_sync(0xffffffffu, o_lo, st, G) - base, hi = __shfl_sync(0xffffffffu, o_hi, st, G) - base;
    double sum = 0.0;
    if (st < c)
      for (int i = lo + sub; i < hi; i += gp) sum += xbuf[i].x;
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const double v = __shfl_xor_sync(0xffffffffu, sum, o, G);
      if (o < gp) sum += v;
    }
    bool bad = false;
    double val = 0.0;
    if (st < c && sub == 0) {
      const int s = s0 + st;
      double fin = neg_inf();
      if (!FWD) {
        const double fc = final_cost(b.fin_g[s], b.fin_a[s], a.cp);
        if (fc < pos_inf() && !(BEAM && final_pruned(a, l, s, fc))) {
          fin = -fc;
          sum += fast_exp(fin - ref);
        }
      }
      const int terms = hi - lo + (fin > neg_inf() ? 1 : 0);
      if (terms <= 2) {
        // one or two terms: exactly Kaldi's LogAdd (x, or max + log1p(exp(-|d|))), so
        // chains and diamonds reproduce the reference bit for bit
        val = fin;
        for (int i = lo; i < hi; ++i) {
          const int4 r = __ldg(rec + base + i);
          double x = score[r.x] - rec_cost(r, a.cp);
          if (BEAM && sweep_arc_pruned<FWD, BEAM>(a, l, base + i, r)) x = neg_inf();
          val = log_add(val, x);
        }
      } else if (sum >= 1e-280 && sum <= 1e280) {
        val = ref + fast_log(sum);
      } else {
        bad = true;
      }
      if (bad) val = sweep_state_exact<FWD, BEAM>(a, l, s);
      score[s] = val;
      ring[s & (kRing - 1)] = val;
    }
    if (!done && c == 0 && sl == 0) {  // a single state with more arcs than the tile stages
      val = sweep_state_exact<FWD, BEAM>(a, l, s0);
      score[s0] = val;
      ring[s0 & (kRing - 1)] = val;
    }
    // the next reference point: this batch's first state (lane 0 of the tile holds it)
    const double v0 = __shfl_sync(0xffffffffu, val, 0, G);
    if (!done && v0 > neg_inf() && v0 < pos_inf()) ref = v0;
    // ---- advance: next batch, next level, or finished
    if (!done) {
      s0 += c > 0 ? c : 1;
      if (s0 >= a1) {
        if (!FWD && a1 - a0 > kRing) wide = a0;
        j += FWD ? 1 : -1;
        if (FWD ? j >= nl : j < 0) {
          done = true;
        } else {
          s0 = a0 = lv[j];
          a1 = lv[j + 1];
        }
      }
    }
    __syncwarp();
  }
}

// Work queue: unit t < ceil(L / NG) sweeps lattices order[t*NG .. t*NG+NG) forward,
// the following units sweep them backward (a warp's tiles share the direction, so
// they share the code path).
template <int G, bool BEAM>
__global__ void __launch_bounds__(128) k_log_sweeps(const __grid_constant__ SweepArgs a) {
  constexpr int NG = 32 / G;
  __shared__ double2 xs[4][kSweepCapPerLane * 32];
  __shared__ double rings[4][NG * sweep_ring(G)];
  const int lane = threadIdx.x & 31;
  double2* xwarp = xs[threadIdx.x >> 5];
  double* rwarp = rings[threadIdx.x >> 5];
  const int per_dir = (a.b.L + NG - 1) / NG;
  const int nunits = per_dir * (a.do_fwd + a.do_bwd);
  for (;;) {
    int unit = 0;
    if (lane == 0) unit = atomicAdd(a.counter, 1);
    unit = __shfl_sync(0xffffffffu, unit, 0);
    if (unit >= nunits) break;
    const bool fwd = a.do_fwd && unit < per_dir;
    const int first = (unit - (fwd || !a.do_fwd ? 0 : per_dir)) * NG;
    if (fwd) log_sweep_tiles<G, true, BEAM>(a, first, lane, xwarp, rwarp);
    else log_sweep_tiles<G, false, BEAM>(a, first, lane, xwarp, rwarp);
    __syncwarp();
  }
}

// total = 0.5 * (tot_forward + beta[start]) as ComputeLatticeAlphasAndBetas
// returns it; tot_forward folds the final states in ascending packed order.
template <bool BEAM>
__global__ void k_totals(SweepArgs a, double* total, double* totfwd) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= a.b.L) return;
  const int l = warp;
  const int s0 = a.b.s_off[l], s1 = a.b.s_off[l + 1];
  if (s0 == s1) {
    if (lane == 0) {
      total[l] = 0.0;
      totfwd[l] = 0.0;
    }
    return;
  }
  double acc = neg_inf();
  for (int s = s0 + lane; s < s1; s += 32) {
    const float fg = a.b.fin_g[s], fa = a.b.fin_a[s];
    if (isinf(fg) && isinf(fa)) continue;
    const double fc = final_cost(fg, fa, a.cp);
    if (BEAM && final_pruned(a, l, s, fc)) continue;
    acc = log_add(acc, a.alpha[s] - fc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc = log_add(acc, __shfl_xor_sync(0xffffffffu, acc, o));
  if (lane == 0) {
    totfwd[l] = acc;
    total[l] = 0.5 * (acc + a.beta[s0]);
  }
}

// ---------------------------------------------------------------- tropical ---
template <int G>
__device__ void trop_forward(const SweepArgs& a, double* vfwd, double* best, int l, int lane) {
  const BatchView& b = a.b;
  const int s_begin = b.s_off[l], s_end = b.s_off[l + 1];
  if (s_begin == s_end) {
    if (lane == 0) best[l] = pos_inf();
    return;
  }
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  for (int s = lv[0] + lane; s < lv[1]; s += 32) vfwd[s] = (s == s_begin) ? 0.0 : pos_inf();
  __syncwarp();
  constexpr int SPW = 32 / G;
  const int grp = lane / G, sl = lane % G;
  for (int j = 1; j < nl; ++j) {
    const int a0 = lv[j], a1 = lv[j + 1];
    for (int base = a0; base < a1; base += SPW) {
      const int s = base + grp;
      const bool act = s < a1;
      const int e0 = act ? b.in_off[s] : 0, e1 = act ? b.in_off[s + 1] : 0;
      double m = pos_inf();
      for (int e = e0 + sl; e < e1; e += G) {
        const int4 r = __ldg(b.in_rec + e);
        m = fmin(m, __dadd_rn(vfwd[r.x], rec_cost(r, a.cp)));
      }
      m = group_min<G>(m);
      if (act && sl == 0) vfwd[s] = m;
    }
    __syncwarp();
  }
  // best_final_cost = min_s fwd[s] + final(s)
  double bf = pos_inf();
  for (int s = s_begin + lane; s < s_end; s += 32)
    bf = fmin(bf, __dadd_rn(vfwd[s], final_cost(b.fin_g[s], b.fin_a[s], a.cp)));
  bf = group_min<32>(bf);
  if (lane == 0) best[l] = bf;
}

template <int G>
__device__ void trop_backward(const SweepArgs& a, double* vbwd, int l, int lane) {
  const BatchView& b = a.b;
  const int s_begin = b.s_off[l], s_end = b.s_off[l + 1];
  if (s_begin == s_end) return;
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  constexpr int SPW = 32 / G;
  const int grp = lane / G, sl = lane % G;
  for (int j = nl - 1; j >= 0; --j) {
    const int a0 = lv[j], a1 = lv[j + 1];
    for (int base = a0; base < a1; base += SPW) {
      const int s = base + grp;
      const bool act = s < a1;
      const int e0 = act ? b.out_off[s] : 0, e1 = act ? b.out_off[s + 1] : 0;
      double m = pos_inf();
      if (act && sl == 0) m = final_cost(b.fin_g[s], b.fin_a[s], a.cp);
      for (int e = e0 + sl; e < e1; e += G) {
        const int4 r = __ldg(b.out_rec + e);
        m = fmin(m, __dadd_rn(rec_cost(r, a.cp), vbwd[r.x]));
      }
      m = group_min<G>(m);
      if (act && sl == 0) vbwd[s] = m;
    }
    __syncwarp();
  }
}

template <int G>
__global__ void __launch_bounds__(128) k_trop_sweeps(SweepArgs a, double* vfwd, double* vbwd, double* best) {
  const int lane = threadIdx.x & 31;
  const int nitems = a.b.L * 2;
  for (;;) {
    int item = 0;
    if (lane == 0) item = atomicAdd(a.counter, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= nitems) break;
    const int l = a.b.order[item >> 1];
    if ((item & 1) == 0) trop_forward<G>(a, vfwd, best, l, lane);
    else trop_backward<G>(a, vbwd, l, lane);
  }
}

// ------------------------------------------------------------- banded log ---
// alpha2[band_off[s] + (len - band_lo[s])] = log-sum of all paths start -> s that
// carry exactly `len` non-epsilon labels: the forward scores of the lattice that
// DisambiguateStateInputSequenceLength (fstext/fstext-utils2.h:109-215) unfolds,
// without unfolding it.
//
// One CTA owns one lattice (work queue).  A level's cells -- (state, len) pairs, a
// contiguous run of the band array -- are spread over the threads with consecutive
// threads on consecutive lengths, so the predecessor's scores are read as contiguous
// runs.  Per level (cut into pieces of <= kBandStates states / kBandArcs arcs) the
// incoming arcs are staged once in shared memory as {cost, where the source's band
// starts relative to the length axis, its valid length range}: a cell's inner loop is
// two shared-memory reads, a range test and one coalesced global read per arc.
// Sums of one or two terms are Kaldi's LogAdd exactly; longer ones a streaming
// log-sum-exp (one exp per term).
constexpr int kBandThreads = 512;
constexpr int kBandArcs = 768;
constexpr int kBandStates = 128;

struct LogSumRun {  // streaming log-sum-exp that remembers its first two terms
  double m, s, x1, x2;
  int n;
  __device__ LogSumRun() : m(neg_inf()), s(0.0), x1(neg_inf()), x2(neg_inf()), n(0) {}
  __device__ __forceinline__ void add(double v) {
    if (v == neg_inf()) return;
    if (n == 0) x1 = v;
    else if (n == 1) x2 = v;
    ++n;
    if (v <= m) {
      s += fast_exp(v - m);
    } else {
      s = (m == neg_inf() ? 0.0 : s * fast_exp(m - v)) + 1.0;
      m = v;
    }
  }
  __device__ __forceinline__ double value() const {
    if (n == 0) return neg_inf();
    if (n == 1) return x1;
    if (n == 2) return log_add(x1, x2);
    return m + fast_log(s);
  }
};

template <bool BEAM>
__global__ void __launch_bounds__(kBandThreads) k_banded_alpha(SweepArgs a, double* alpha2_chunk, int l0, int l1,
                                                                long long band_base) {
  __shared__ double sa_cost[kBandArcs];
  __shared__ long long sa_base[kBandArcs];
  __shared__ int2 sa_range[kBandArcs];
  __shared__ int ss_arc[kBandStates + 1];
  __shared__ long long ss_cell[kBandStates + 1];
  __shared__ int ss_lo[kBandStates];
  __shared__ int s_item, s_take;
  double* alpha2 = alpha2_chunk - band_base;  // indexed with global band offsets
  const BatchView& b = a.b;
  const int tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_item = atomicAdd(a.counter, 1);
    __syncthreads();
    if (s_item >= l1 - l0) break;
    const int l = l0 + s_item;
    const int s_begin = b.s_off[l], s_end = b.s_off[l + 1];
    if (s_begin == s_end) continue;
    const int* lv = b.lvl_start + b.lvl_off[l];
    const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
    // level 0: the start state has the single cell (len 0) = 0; other sources are unreachable (width 0)
    for (int s = lv[0] + tid; s < lv[1]; s += kBandThreads)
      if (s == s_begin && b.band_off[s + 1] > b.band_off[s]) alpha2[b.band_off[s]] = 0.0;
    for (int j = 1; j < nl; ++j) {
      const int a1 = lv[j + 1];
      int s0 = lv[j];
      while (s0 < a1) {
        __syncthreads();  // the previous piece's cells are written, its staging arrays free
        // ---- the piece: states [s0, s0 + take), as many as fit the staging arrays (>= 1)
        const int nst = min(a1 - s0, kBandStates);
        for (int k = tid; k <= nst; k += kBandThreads) {
          ss_arc[k] = b.in_off[s0 + k];
          ss_cell[k] = b.band_off[s0 + k];
          if (k < nst) ss_lo[k] = b.band_lo[s0 + k];
        }
        if (tid == 0) s_take = 1;
        __syncthreads();
        const int e_base = ss_arc[0];
        for (int k = tid + 1; k <= nst; k += kBandThreads)
          if (ss_arc[k] - e_base <= kBandArcs) atomicMax(&s_take, k);
        __syncthreads();
        const int take = s_take;
        const int narcs = ss_arc[take] - e_base;
        const bool staged = narcs <= kBandArcs;  // else: one state with more arcs than fit (take == 1)
        if (staged) {
          for (int i = tid; i < narcs; i += kBandThreads) {
            const int4 r = __ldg(b.in_rec + e_base + i);
            const int plo = b.band_lo[r.x];
            const int pw = (int)(b.band_off[r.x + 1] - b.band_off[r.x]);
            const int nz = r.w != 0 ? 1 : 0;
            bool dead = plo < 0 || pw <= 0;
            if (BEAM && !dead) {
              const int lo = last_le(ss_arc, 0, take - 1, e_base + i);  // the arc's destination: last k with ss_arc[k] <= e
              dead = arc_pruned(a, l, r.x, s0 + lo, r);
            }
            sa_cost[i] = rec_cost(r, a.cp);
            sa_base[i] = b.band_off[r.x] - plo - nz;           // cell of (source, len - nz) = base + len
            sa_range[i] = dead ? make_int2(0, 0) : make_int2(plo + nz, plo + pw + nz);  // valid len: [x, y)
          }
        }
        __syncthreads();
        const long long c0 = ss_cell[0], c1 = ss_cell[take];
        for (long long cell = c0 + tid; cell < c1; cell += kBandThreads) {
          const int lo = last_le(ss_cell, 0, take - 1, cell);  // last k with ss_cell[k] <= cell
          const int len = ss_lo[lo] + (int)(cell - ss_cell[lo]);
          LogSumRun acc;
          if (staged) {
            // ONE pass over the state's staged arcs: the exp terms are taken around alpha[s] of the
            // plain sweep (run just before), which bounds every term from above -- alpha[s] is the
            // log-sum over all lengths of what this cell sums for one -- so no maximum has to be
            // found first; two accumulators, no loop-carried chain longer than one add.  The first
            // two finite terms are kept for Kaldi's exact LogAdd; a sum that leaves [1e-280, 1e280]
            // (a cell more than ~645 nats below alpha[s], or inconsistent scores) is redone around
            // its own maximum.
            const int i0 = ss_arc[lo] - e_base, i1 = ss_arc[lo + 1] - e_base;
            const double ref = a.alpha[s0 + lo];
            double sum0 = 0.0, sum1 = 0.0;
            int nterm = 0;
            {
              int i = i0;
              for (; i + 1 < i1; i += 2) {  // branch-free: exp(-inf) = 0 for the arcs that do not reach this length
                const int2 ra = sa_range[i], rb = sa_range[i + 1];
                const double xa = (len >= ra.x && len < ra.y) ? alpha2[sa_base[i] + len] - sa_cost[i] : neg_inf();
                const double xb = (len >= rb.x && len < rb.y) ? alpha2[sa_base[i + 1] + len] - sa_cost[i + 1] : neg_inf();
                nterm += (xa > neg_inf() ? 1 : 0) + (xb > neg_inf() ? 1 : 0);
                sum0 += fast_exp(xa - ref);
                sum1 += fast_exp(xb - ref);
              }
              if (i < i1) {
                const int2 ra = sa_range[i];
                const double xa = (len >= ra.x && len < ra.y) ? alpha2[sa_base[i] + len] - sa_cost[i] : neg_inf();
                nterm += xa > neg_inf() ? 1 : 0;
                sum0 += fast_exp(xa - ref);
              }
            }
            if (nterm >= 3) {
              const double ssum = sum0 + sum1;
              if (ssum >= 1e-280 && ssum <= 1e280) {
                alpha2[cell] = ref + fast_log(ssum);
                continue;
              }
              double m = neg_inf();  // rare: around the cell's own maximum
              for (int i = i0; i < i1; ++i) {
                const int2 rg = sa_range[i];
                if (len >= rg.x && len < rg.y) m = fmax(m, alpha2[sa_base[i] + len] - sa_cost[i]);
              }
              double sum = 0.0;
              for (int i = i0; i < i1; ++i) {
                const int2 rg = sa_range[i];
                if (len >= rg.x && len < rg.y) sum += fast_exp(alpha2[sa_base[i] + len] - sa_cost[i] - m);
              }
              alpha2[cell] = m + fast_log(sum);
              continue;
            }
            if (nterm > 0)  // one or two terms: Kaldi's LogAdd exactly
              for (int i = i0; i < i1; ++i) {
                const int2 rg = sa_range[i];
                if (len >= rg.x && len < rg.y) acc.add(alpha2[sa_base[i] + len] - sa_cost[i]);
              }
          } else {
            const int s = s0 + lo;
            for (int e = b.in_off[s]; e < b.in_off[s + 1]; ++e) {
              const int4 r = __ldg(b.in_rec + e);
              const int plen = len - (r.w != 0 ? 1 : 0);
              const int plo = b.band_lo[r.x];
              const int pw = (int)(b.band_off[r.x + 1] - b.band_off[r.x]);
              if (plo < 0 || plen < plo || plen >= plo + pw) continue;
              if (BEAM && arc_pruned(a, l, r.x, s, r)) continue;
              acc.add(alpha2[b.band_off[r.x] + plen - plo] - rec_cost(r, a.cp));
            }
          }
          alpha2[cell] = acc.value();
        }
        s0 += take;
      }
    }
  }
}

int sweep_grid(klu_ctx* c, int items) {
  const int warps_per_block = 4;
  const int max_blocks = c->num_sms * 16;  // 64 resident warps per SM
  int blocks = (items + warps_per_block - 1) / warps_per_block;
  return std::max(1, std::min(blocks, max_blocks));
}

SweepArgs make_args(klu_ctx* c, const CostParams& cp, bool use_beam, float beam) {
  SweepArgs a;
  a.b = c->view();
  a.cp = cp;
  a.alpha = c->d_alpha.as<double>();
  a.beta = c->d_beta.as<double>();
  a.vfwd = use_beam ? c->d_vfwd.as<double>() : nullptr;
  a.vbwd = use_beam ? c->d_vbwd.as<double>() : nullptr;
  a.best = use_beam ? c->d_best.as<double>() : nullptr;
  a.beam = (double)beam;
  a.counter = c->d_counter.as<int>();
  a.do_fwd = 1;
  a.do_bwd = 1;
  return a;
}

}  // namespace

int pick_group(double avg_deg) {
  if (avg_deg <= 3.0) return 2;
  if (avg_deg <= 6.0) return 4;
  if (avg_deg <= 48.0) return 8;
  if (avg_deg <= 160.0) return 16;
  return 32;
}

int run_log_sweeps(klu_ctx* c, const CostParams& cp, bool use_beam, float beam) {
  KLU_TRY(c->d_alpha.reserve(sizeof(double) * std::max<int64_t>(c->S, 1)));
  KLU_TRY(c->d_beta.reserve(sizeof(double) * std::max<int64_t>(c->S, 1)));
  KLU_TRY(c->d_total.reserve(sizeof(double) * std::max<int32_t>(c->L, 1)));
  KLU_TRY(c->d_totfwd.reserve(sizeof(double) * std::max<int32_t>(c->L, 1)));
  KLU_TRY(c->d_counter.reserve(64));
  if (c->L == 0) return 0;
  KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));
  SweepArgs a = make_args(c, cp, use_beam, beam);
  // lanes per lattice: enough to stream a level's arcs in ~5 trips (measured best on
  // 80-arc levels: 16), more when there are too few lattices to fill the machine otherwise
  int G = 4;
  {
    const double arcs_per_level = c->NL > 0 ? (double)c->E / (double)c->NL : 1.0;
    while (G < 32 && G * 6 < arcs_per_level) G <<= 1;
    while (G < 32 && (int64_t)2 * c->L * G / 32 < (int64_t)c->num_sms * 8) G <<= 1;
    if (const char* env = getenv("KLU_SWEEP_LANES")) G = atoi(env);
  }
  const int units = 2 * ((c->L + 32 / G - 1) / (32 / G));
  const int grid = sweep_grid(c, units);
  {
    KLU_LAUNCH(c, "k_log_sweeps");
    KLU_DISPATCH_G(G, if (use_beam) k_log_sweeps<kG, true><<<grid, 128, 0, c->stream>>>(a);
                   else k_log_sweeps<kG, false><<<grid, 128, 0, c->stream>>>(a));
  }
  KLU_TRY(check_launch("k_log_sweeps"));
  {
    KLU_LAUNCH(c, "k_totals");
    const int blocks = (c->L * 32 + 127) / 128;
    if (use_beam) k_totals<true><<<blocks, 128, 0, c->stream>>>(a, c->d_total.as<double>(), c->d_totfwd.as<double>());
    else k_totals<false><<<blocks, 128, 0, c->stream>>>(a, c->d_total.as<double>(), c->d_totfwd.as<double>());
  }
  return check_launch("k_totals");
}

int run_tropical_sweeps(klu_ctx* c, const CostParams& cp) {
  KLU_TRY(c->d_vfwd.reserve(sizeof(double) * std::max<int64_t>(c->S, 1)));
  KLU_TRY(c->d_vbwd.reserve(sizeof(double) * std::max<int64_t>(c->S, 1)));
  KLU_TRY(c->d_best.reserve(sizeof(double) * std::max<int32_t>(c->L, 1)));
  KLU_TRY(c->d_counter.reserve(64));
  if (c->L == 0) return 0;
  KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));
  SweepArgs a = make_args(c, cp, false, 0.f);
  const int G = pick_group(c->avg_deg);
  const int grid = sweep_grid(c, c->L * 2);
  {
    KLU_LAUNCH(c, "k_trop_sweeps");
    KLU_DISPATCH_G(G, k_trop_sweeps<kG><<<grid, 128, 0, c->stream>>>(a, c->d_vfwd.as<double>(),
                                                                      c->d_vbwd.as<double>(), c->d_best.as<double>()));
  }
  return check_launch("k_trop_sweeps");
}

int run_banded_alpha(klu_ctx* c, const CostParams& cp, bool use_beam, float beam, int l0, int l1) {
  const long long band_base = c->h_band_off[l0];
  const long long cells = c->h_band_off[l1] - band_base;
  KLU_TRY(c->d_alpha2.reserve(sizeof(double) * std::max<long long>(cells, 1)));
  KLU_TRY(c->d_counter.reserve(64));
  if (l1 <= l0) return 0;
  KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));
  SweepArgs a = make_args(c, cp, use_beam, beam);
  const int grid = std::max(1, std::min(l1 - l0, c->num_sms * 8));  // one CTA per lattice in flight
  {
    KLU_LAUNCH(c, "k_banded_alpha");
    if (use_beam) k_banded_alpha<true><<<grid, kBandThreads, 0, c->stream>>>(a, c->d_alpha2.as<double>(), l0, l1, band_base);
    else k_banded_alpha<false><<<grid, kBandThreads, 0, c->stream>>>(a, c->d_alpha2.as<double>(), l0, l1, band_base);
  }
  return check_launch("k_banded_alpha");
}

}  // namespace klu
