// klu_prune.cu -- lattice-prune-dyn-beam on the GPU (SURVEY.md K9, K10).
//
// Reference: latbin/lattice-prune-dyn-beam.cc:27-90 (ComputeLatticeBeam) and
// :148-207 (the loop `beam *= beam_ratio; PruneLattice(beam)` until the lattice
// has <= max-arcs arcs and <= max-states states or beam <= min-beam, then the
// inverse scaling and the write).
//
// PruneLattice [ext] keeps an arc iff  fwd[s] + (cost + bwd[next]) <= best + beam
// and a final weight iff  final + fwd[s] <= best + beam;  Connect() then drops the
// states no surviving arc or final touches.  fwd, bwd and best of the surviving
// part do not change from one iteration to the next (the best path through any
// surviving arc survives with it), so one tropical forward/backward sweep gives a
// per-arc forward-backward cost once, and the whole loop becomes a search over
// thresholds: per iteration one counting pass over those costs.  Every value is a
// min/max/sum of the same doubles the reference forms, in the same association, so
// the surviving arc set is bit-exact.
#include <math.h>

#include <algorithm>

#include <string.h>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

struct PruneArgs {
  BatchView b;
  CostParams cp;
  const double* vfwd;
  const double* vbwd;
  const double* best;
  double* fb;        // [E] out-order arcs: fwd[s] + (cost + bwd[next])
  double* smin;      // [S] min forward-backward cost over everything touching the state
  double* ffb;       // [S] final + fwd (inf when not final)
  float beam_ratio, min_beam;
  int max_arcs, max_states;
  double* beams;     // [2L] original beam, final beam
  double* cutoff;    // [L] final cutoff (best + (float)beam), only valid when iters > 0
  int* iters;        // [L]
  int* status;       // [L] 1 = loop does not terminate (infinite beam)
  // outputs (input index space)
  int* arc_keep;     // [E] by (lattice e_off + original arc index): 0/1, then exclusive scan
  int* state_keep;   // [S] by (lattice s_off + original state id): 0/1, then exclusive scan
  int* arc_cnt;      // [L]
  int* state_cnt;    // [L]
  const int64_t* res_off;  // [L+1]
  int32_t *o_arc, *o_src, *o_dst;
  float *o_g, *o_a;
  int32_t* o_smap;   // [S] input numbering
  float *o_fg, *o_fa;
  double inv_gs, inv_as;
};

// per out-order arc: forward-backward cost
__global__ void __launch_bounds__(256) k_prune_fb(PruneArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < a.b.E; e += stride) {
    const int4 r = a.b.out_rec[e];
    const int s = a.b.out_src[e];
    a.fb[e] = __dadd_rn(a.vfwd[s], __dadd_rn(rec_cost(r, a.cp), a.vbwd[r.x]));
  }
}

// per state: final fb and the smallest fb over final, outgoing and incoming arcs
__global__ void __launch_bounds__(256) k_prune_smin(PruneArgs a) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < a.b.S; s += stride) {
    const double fc = final_cost(a.b.fin_g[s], a.b.fin_a[s], a.cp);
    const double ffb = fc == pos_inf() ? pos_inf() : __dadd_rn(fc, a.vfwd[s]);
    // min over outgoing arcs and the final weight = fwd + bwd (addition is monotone)
    double m = fmin(ffb, __dadd_rn(a.vfwd[s], a.vbwd[s]));
    for (int e = a.b.in_off[s]; e < a.b.in_off[s + 1]; ++e) {
      const int4 r = a.b.in_rec[e];
      m = fmin(m, __dadd_rn(a.vfwd[r.x], __dadd_rn(rec_cost(r, a.cp), a.vbwd[s])));
    }
    a.ffb[s] = ffb;
    a.smin[s] = m;
  }
}

__device__ __forceinline__ double block_max(double v, double* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  double r = sh[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmax(r, sh[w]);
  return r;
}

__device__ __forceinline__ int block_sum(int v, int* sh) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  int r = 0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) r += sh[w];
  return r;
}

// One CTA per lattice: ComputeLatticeBeam, then the dynamic-beam loop as a
// threshold search.
__global__ void __launch_bounds__(256) k_prune_search(PruneArgs a) {
  __shared__ double shd[8];
  __shared__ int shi[8];
  const int l = blockIdx.x;
  const int s0 = a.b.s_off[l], s1 = a.b.s_off[l + 1];
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const int tid = threadIdx.x;
  if (s0 == s1) {
    if (tid == 0) {
      a.beams[2 * l] = 0.0;  // ComputeLatticeBeam returns 0 for an empty lattice, :34
      a.beams[2 * l + 1] = 0.0;
      a.iters[l] = 0;
      a.status[l] = 0;
      a.cutoff[l] = 0.0;
    }
    return;
  }
  const double best = a.best[l];
  // cutoff = max(best, finite-final fb, arc fb), :60-87
  double mx = best;
  for (int e = e0 + tid; e < e1; e += 256) mx = fmax(mx, a.fb[e]);
  for (int s = s0 + tid; s < s1; s += 256) {
    const double fc = final_cost(a.b.fin_g[s], a.b.fin_a[s], a.cp);
    if (fc != pos_inf()) mx = fmax(mx, a.ffb[s]);
  }
  mx = block_max(mx, shd);
  const double beam0 = mx - best;
  double beam = beam0;
  int num_arcs = e1 - e0, num_states = s1 - s0;
  int n = 0;
  double cut = 0.0;
  const double min_beam = (double)a.min_beam;
  int bad = 0;
  while (beam > min_beam && (num_arcs > a.max_arcs || num_states > a.max_states)) {
    if (n >= 1000000 || !(beam < pos_inf())) {  // the reference would never leave this loop
      bad = 1;
      break;
    }
    beam = (double)a.beam_ratio * beam;  // float * double, :170
    cut = __dadd_rn(best, (double)(float)beam);  // PruneLattice(BaseFloat beam): cutoff = best + beam
    int ca = 0, cs = 0;
    for (int e = e0 + tid; e < e1; e += 256) ca += !(a.fb[e] > cut);
    for (int s = s0 + tid; s < s1; s += 256) cs += !(a.smin[s] > cut);
    num_arcs = block_sum(ca, shi);
    num_states = block_sum(cs, shi);
    ++n;
  }
  if (tid == 0) {
    a.beams[2 * l] = beam0;
    a.beams[2 * l + 1] = beam;
    a.iters[l] = n;
    a.cutoff[l] = cut;
    a.status[l] = bad;
  }
}

// keep flags in the caller's index space
__global__ void __launch_bounds__(256) k_prune_mark(PruneArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int s0 = a.b.s_off[l], s1 = a.b.s_off[l + 1];
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const bool all = a.iters[l] == 0;
  const double cut = a.cutoff[l];
  const int t = lt.tile * blockDim.x + threadIdx.x, stride = lt.tiles * blockDim.x;
  for (int e = e0 + t; e < e1; e += stride) a.arc_keep[e0 + a.b.out_orig[e]] = (all || !(a.fb[e] > cut)) ? 1 : 0;
  for (int s = s0 + t; s < s1; s += stride) a.state_keep[s0 + a.b.orig[s]] = (all || !(a.smin[s] > cut)) ? 1 : 0;
}

// One CTA per lattice: exclusive scans of both flag arrays (in place) + counts.
__global__ void __launch_bounds__(256) k_prune_scan(PruneArgs a) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = blockIdx.x;
  const int tid = threadIdx.x;
  for (int which = 0; which < 2; ++which) {
    int* flags = which == 0 ? a.arc_keep : a.state_keep;
    const int i0 = which == 0 ? a.b.e_off[l] : a.b.s_off[l];
    const int i1 = which == 0 ? a.b.e_off[l + 1] : a.b.s_off[l + 1];
    __syncthreads();
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (int tile = i0; tile < i1; tile += 256) {
      const int i = tile + tid;
      const int c = i < i1 ? flags[i] : 0;
      const int pre = cta_exclusive_scan<int, 256>(c, warp_sum, carry_s);
      // exclusive rank, sign bit marks "dropped"
      if (i < i1) flags[i] = c ? pre : -1;
    }
    if (tid == 0) (which == 0 ? a.arc_cnt : a.state_cnt)[l] = carry_s;
  }
}

// Output weights: scale -> (+penalty) -> [prune] -> inverse scale -> (-penalty),
// each step rounded to float exactly where the reference stores a float (:188-192).
__device__ __forceinline__ void out_weights(float g, float w, int label, const PruneArgs& a, float* go, float* ao) {
  float g2, a2;
  scaled_weights(g, w, label, a.cp, &g2, &a2);
  if (a.cp.scale && !(isinf(g2) && isinf(a2) && g2 > 0 && a2 > 0)) {
    g2 = (float)__dmul_rn(a.inv_gs, (double)g2);
    a2 = (float)__dmul_rn(a.inv_as, (double)a2);
  }
  if (label != 0) g2 = __fadd_rn(g2, -a.cp.pen);
  *go = g2;
  *ao = a2;
}

__global__ void __launch_bounds__(256) k_prune_emit(PruneArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int s0 = a.b.s_off[l], s1 = a.b.s_off[l + 1];
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const int64_t out = a.res_off[l];
  const bool all = a.iters[l] == 0;
  const double cut = a.cutoff[l];
  const int t = lt.tile * blockDim.x + threadIdx.x, stride = lt.tiles * blockDim.x;
  for (int e = e0 + t; e < e1; e += stride) {
    const int o = a.b.out_orig[e];
    const int pos = a.arc_keep[e0 + o];
    if (pos < 0) continue;
    const int4 r = a.b.out_rec[e];
    const int s = a.b.out_src[e];
    a.o_arc[out + pos] = o;
    a.o_src[out + pos] = a.state_keep[s0 + a.b.orig[s]];
    a.o_dst[out + pos] = a.state_keep[s0 + a.b.orig[r.x]];
    float g, w;
    out_weights(__int_as_float(r.y), __int_as_float(r.z), r.w, a, &g, &w);
    a.o_g[out + pos] = g;
    a.o_a[out + pos] = w;
  }
  for (int s = s0 + t; s < s1; s += stride) {
    const int os = s0 + a.b.orig[s];
    a.o_smap[os] = a.state_keep[os];
    float g = a.b.fin_g[s], w = a.b.fin_a[s];
    const bool is_final = !(isinf(g) && isinf(w));
    bool keep_final = is_final;
    if (is_final && !all) keep_final = !(a.ffb[s] > cut);  // SetFinal(state, Zero) in PruneLattice
    if (keep_final) out_weights(g, w, 0, a, &g, &w);
    a.o_fg[os] = keep_final ? g : INFINITY;
    a.o_fa[os] = keep_final ? w : INFINITY;
  }
}

// ----------------------------------------------------------- lattice-prune-arcs ---
// latbin/lattice-prune-arcs.cc:34-84 (SURVEY.md 8f rank 4).  As written there: arcs sorted by
// ascending cost-through = cost_arc - alpha[s] - beta[next] (most probable first), their mass
// accumulated in that order until -log(mass) < beam - total, and the arcs FROM that one on put
// back with AddArc (so a state's arcs come back in sorted order); Connect [ext] trims the rest.
// The source's std::sort compares the cost alone, so arcs of EQUAL cost have no defined order
// there; here they keep the lattice's own arc order (a stable sort -- one of its valid outcomes).
struct PruneArcsArgs {
  const double* alpha;
  const double* beta;
  const double* total;
  double beam;
  const int64_t* seg_base;  // [L] = e_off
  const int32_t* seg_cnt;   // [L]
  unsigned long long *key_a, *key_b;
  unsigned int *idx_a, *idx_b;
  const unsigned char* where;
  int* first_kept;      // [L] rank of the first arc put back (== arcs: nothing is)
  int* rank;            // [E] by (e_off + original arc index): position in the sorted order
  unsigned char* reach; // [S] packed states: bit 0 accessible, bit 1 co-accessible over the kept arcs
};

// grid (lattices, tiles): sort key of every arc, laid out in the caller's arc order (the
// stable sort then breaks ties by that order)
__global__ void __launch_bounds__(256) k_pa_keys(PruneArgs a, PruneArcsArgs p) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  for (int e = e0 + lt.tile * blockDim.x + threadIdx.x; e < e1; e += lt.tiles * blockDim.x) {
    const int4 r = a.b.out_rec[e];
    const int s = a.b.out_src[e];
    const int o = a.b.out_orig[e];
    // cost_arc + alphas[s] + betas[nextstate] with both vectors negated, :52-53
    const double ct = __dadd_rn(__dadd_rn(rec_cost(r, a.cp), -p.alpha[s]), -p.beta[r.x]);
    p.key_a[e0 + o] = ord_f64(ct);
    p.idx_a[e0 + o] = (unsigned int)o;
  }
}

// one thread per lattice: the accumulation loop of :62-69 in sorted order, to the cut
__global__ void __launch_bounds__(128) k_pa_cut(PruneArgs a, PruneArcsArgs p, double* beams) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= a.b.L) return;
  const int n = p.seg_cnt[l];
  const unsigned long long* key = (p.where[l] ? p.key_b : p.key_a) + p.seg_base[l];
  const double cutoff = a.b.s_off[l] == a.b.s_off[l + 1] ? 0.0 : __dadd_rn(p.beam, -p.total[l]);
  double cost_acc = pos_inf();
  int i = 0;
  for (; i < n; ++i) {
    const unsigned long long k = key[i];
    const unsigned long long bits = (k & 0x8000000000000000ULL) ? (k & 0x7fffffffffffffffULL) : ~k;  // ord_f64 inverted
    const double ct = __longlong_as_double((long long)bits);
    cost_acc = -log_add(-cost_acc, -ct);
    if (cost_acc < cutoff) break;
  }
  p.first_kept[l] = i;
  beams[2 * l] = cutoff;
  beams[2 * l + 1] = (double)i;
}

// grid (lattices, tiles): rank of every arc in the sorted order, by original arc index
__global__ void __launch_bounds__(256) k_pa_rank(PruneArgs a, PruneArcsArgs p) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int n = p.seg_cnt[l];
  const int e0 = a.b.e_off[l];
  const unsigned int* idx = (p.where[l] ? p.idx_b : p.idx_a) + p.seg_base[l];
  for (int q = lt.tile * blockDim.x + threadIdx.x; q < n; q += lt.tiles * blockDim.x) p.rank[e0 + (int)idx[q]] = q;
}

// One warp per lattice: fst::Connect over the arcs put back -- accessible from the start
// (forward over the levels), co-accessible to a final state (backward) -- then the keep flags
// in the caller's index space.
__global__ void __launch_bounds__(128) k_pa_connect(PruneArgs a, PruneArcsArgs p) {
  const int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (l >= a.b.L) return;
  const BatchView& b = a.b;
  const int s0 = b.s_off[l], s1 = b.s_off[l + 1];
  const int e0 = b.e_off[l], e1 = b.e_off[l + 1];
  if (s0 == s1) return;
  const int first = p.first_kept[l];
  const bool none = first >= e1 - e0;  // nothing put back: DeleteStates(), :71-73
  const int* lv = b.lvl_start + b.lvl_off[l];
  const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
  for (int s = s0 + lane; s < s1; s += 32) p.reach[s] = (!none && s == s0) ? 1 : 0;
  __syncwarp();
  for (int j = 1; j < nl && !none; ++j) {
    for (int s = lv[j] + lane; s < lv[j + 1]; s += 32) {
      unsigned char r = 0;
      for (int e = b.in_off[s]; e < b.in_off[s + 1] && !r; ++e) {
        const int src = b.in_rec[e].x;
        if (p.rank[e0 + b.out_orig[b.in2out[e]]] >= first && (p.reach[src] & 1)) r = 1;
      }
      p.reach[s] = r;
    }
    __syncwarp();
  }
  for (int j = nl - 1; j >= 0 && !none; --j) {
    for (int s = lv[j] + lane; s < lv[j + 1]; s += 32) {
      const float fg = b.fin_g[s], fa = b.fin_a[s];
      unsigned char r = !(isinf(fg) && isinf(fa)) ? 2 : 0;
      for (int e = b.out_off[s]; e < b.out_off[s + 1] && !r; ++e)
        if (p.rank[e0 + b.out_orig[e]] >= first && (p.reach[b.out_rec[e].x] & 2)) r = 2;
      p.reach[s] |= r;
    }
    __syncwarp();
  }
  const bool start_ok = !none && p.reach[s0] == 3;  // Connect deletes everything when the start is not kept
  for (int s = s0 + lane; s < s1; s += 32) a.state_keep[s0 + b.orig[s]] = (start_ok && p.reach[s] == 3) ? 1 : 0;
  __syncwarp();
  for (int e = e0 + lane; e < e1; e += 32) {
    const int o = b.out_orig[e];
    const bool keep = start_ok && p.rank[e0 + o] >= first && p.reach[b.out_src[e]] == 3 && p.reach[b.out_rec[e].x] == 3;
    a.arc_keep[e0 + o] = keep ? 1 : 0;
  }
}

// grid (lattices, tiles): the lattice that is written.  arc_keep / state_keep hold exclusive ranks
// in the caller's order (k_prune_scan); a state's arcs come out in sorted (cost) order, as AddArc
// appended them.
__global__ void __launch_bounds__(256) k_pa_emit(PruneArgs a, PruneArcsArgs p) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const BatchView& b = a.b;
  const int s0 = b.s_off[l], s1 = b.s_off[l + 1];
  const int e0 = b.e_off[l], e1 = b.e_off[l + 1];
  const int64_t out = a.res_off[l];
  const int t = lt.tile * blockDim.x + threadIdx.x, stride = lt.tiles * blockDim.x;
  for (int e = e0 + t; e < e1; e += stride) {
    const int o = b.out_orig[e];
    if (a.arc_keep[e0 + o] < 0) continue;
    const int s = b.out_src[e];
    const int mine = p.rank[e0 + o];
    int base = 0x7fffffff, before = 0;
    for (int q = b.out_off[s]; q < b.out_off[s + 1]; ++q) {  // the state's kept arcs (a contiguous run of ranks)
      const int oq = b.out_orig[q];
      const int kq = a.arc_keep[e0 + oq];
      if (kq < 0) continue;
      base = min(base, kq);
      before += p.rank[e0 + oq] < mine ? 1 : 0;
    }
    const int pos = base + before;
    const int4 r = b.out_rec[e];
    a.o_arc[out + pos] = o;
    a.o_src[out + pos] = a.state_keep[s0 + b.orig[s]];
    a.o_dst[out + pos] = a.state_keep[s0 + b.orig[r.x]];
    float g, w;
    out_weights(__int_as_float(r.y), __int_as_float(r.z), r.w, a, &g, &w);
    a.o_g[out + pos] = g;
    a.o_a[out + pos] = w;
  }
  for (int s = s0 + t; s < s1; s += stride) {
    const int os = s0 + b.orig[s];
    a.o_smap[os] = a.state_keep[os];
    float g = b.fin_g[s], w = b.fin_a[s];
    const bool keep_final = !(isinf(g) && isinf(w)) && a.state_keep[os] >= 0;
    if (keep_final) out_weights(g, w, 0, a, &g, &w);
    a.o_fg[os] = keep_final ? g : INFINITY;
    a.o_fa[os] = keep_final ? w : INFINITY;
  }
}

}  // namespace

int run_prune_arcs(klu_ctx* c, const klu_opts* o) {
  if (!(o->beam > 0.0f)) {
    set_error("--beam_ratio must be in the open range (0.0, inf).");  // latbin/lattice-prune-arcs.cc:131-133 (sic)
    return 1;
  }
  const int32_t L = c->L;
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = 0;
  CostParams cp = make_cost_params(o, false);
  KLU_TRY(run_log_sweeps(c, cp, false, 0.f));
  if (L == 0) return 0;
  const int64_t S = std::max<int64_t>(c->S, 1), E = std::max<int64_t>(c->E, 1);
  enum { P_KEYA = 0, P_KEYB, P_IDXA, P_BEAMS, P_IDXB, P_SEG, P_RANK, P_AKEEP, P_SKEEP, P_ACNT, P_SCNT, P_REACH };
  DevBuf* sc = c->d_scratch;
  KLU_TRY(sc[P_KEYA].reserve(8 * E));
  KLU_TRY(sc[P_KEYB].reserve(8 * E));
  KLU_TRY(sc[P_IDXA].reserve(4 * E));
  KLU_TRY(sc[P_IDXB].reserve(4 * E));
  KLU_TRY(sc[P_BEAMS].reserve(16 * (size_t)L));  // slot 3: klu_fetch_prune reads the beams there
  KLU_TRY(sc[P_SEG].reserve(8 * (size_t)(L + 1) + 4 * (size_t)L + 4 * (size_t)L + (size_t)L + 64));
  KLU_TRY(sc[P_RANK].reserve(4 * E));
  KLU_TRY(sc[P_AKEEP].reserve(4 * E));
  KLU_TRY(sc[P_SKEEP].reserve(4 * S));
  KLU_TRY(sc[P_ACNT].reserve(4 * (size_t)L));
  KLU_TRY(sc[P_SCNT].reserve(4 * (size_t)L));
  KLU_TRY(sc[P_REACH].reserve((size_t)S));
  KLU_TRY(c->d_res[5].reserve(8 * (size_t)(L + 1)));
  for (int i = 0; i < 4; ++i) KLU_TRY(c->d_res[i].reserve(4 * E));
  KLU_TRY(c->d_res[4].reserve(8 * E));
  KLU_TRY(c->d_res[6].reserve(8 * S));
  KLU_TRY(c->d_res[7].reserve(8 * S));
  int64_t* d_seg_base = sc[P_SEG].as<int64_t>();
  int32_t* d_seg_cnt = reinterpret_cast<int32_t*>(d_seg_base + L + 1);
  int* d_first = d_seg_cnt + L;
  unsigned char* d_where = reinterpret_cast<unsigned char*>(d_first + L);
  std::vector<int32_t> seg_cnt(L);
  int64_t max_arcs = 0;
  for (int32_t l = 0; l < L; ++l) {
    seg_cnt[l] = (int32_t)(c->h_e_off[l + 1] - c->h_e_off[l]);
    max_arcs = std::max<int64_t>(max_arcs, seg_cnt[l]);
  }
  KLU_CUDA(cudaMemcpyAsync(d_seg_base, c->h_e_off.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemcpyAsync(d_seg_cnt, seg_cnt.data(), 4 * (size_t)L, cudaMemcpyHostToDevice, c->stream));
  PruneArgs a;
  memset(&a, 0, sizeof(a));
  a.b = c->view();
  a.cp = cp;
  a.arc_keep = sc[P_AKEEP].as<int>();
  a.state_keep = sc[P_SKEEP].as<int>();
  a.arc_cnt = sc[P_ACNT].as<int>();
  a.state_cnt = sc[P_SCNT].as<int>();
  a.res_off = c->d_res[5].as<int64_t>();
  a.o_arc = c->d_res[0].as<int32_t>();
  a.o_src = c->d_res[1].as<int32_t>();
  a.o_dst = c->d_res[2].as<int32_t>();
  a.o_g = c->d_res[3].as<float>();
  a.o_a = c->d_res[4].as<float>();
  a.o_smap = c->d_res[6].as<int32_t>();
  a.o_fg = c->d_res[7].as<float>();
  a.o_fa = c->d_res[7].as<float>() + S;
  a.inv_gs = 1.0 / (double)o->graph_scale;
  a.inv_as = 1.0 / (double)o->acoustic_scale;
  PruneArcsArgs p;
  p.alpha = c->d_alpha.as<double>();
  p.beta = c->d_beta.as<double>();
  p.total = c->d_total.as<double>();
  p.beam = (double)o->beam;
  p.seg_base = d_seg_base;
  p.seg_cnt = d_seg_cnt;
  p.key_a = sc[P_KEYA].as<unsigned long long>();
  p.key_b = sc[P_KEYB].as<unsigned long long>();
  p.idx_a = sc[P_IDXA].as<unsigned int>();
  p.idx_b = sc[P_IDXB].as<unsigned int>();
  p.where = d_where;
  p.first_kept = d_first;
  p.rank = sc[P_RANK].as<int>();
  p.reach = sc[P_REACH].as<unsigned char>();
  const int tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  {
    KLU_LAUNCH(c, "k_pa_keys");
    k_pa_keys<<<dim3(L, tiles), 256, 0, c->stream>>>(a, p);
  }
  KLU_TRY(check_launch("k_pa_keys"));
  SegSortArgs ss;
  ss.seg_base = d_seg_base;
  ss.seg_cnt = d_seg_cnt;
  ss.key_a = p.key_a;
  ss.val_a = p.idx_a;
  ss.key_b = p.key_b;
  ss.val_b = p.idx_b;
  ss.where = d_where;
  ss.lo_bit = 32;  // high half of the f64 keys first, runs that agree there settled afterwards
  ss.hi_bit = 64;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, ss, L, c->E));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(arc costs)"));
  {
    KLU_LAUNCH(c, "k_order_fixup");
    k_seg_order_fixup<<<dim3(L, tiles), 256, 0, c->stream>>>(ss, 0);
  }
  KLU_TRY(check_launch("k_order_fixup"));
  {
    KLU_LAUNCH(c, "k_pa_cut");
    k_pa_cut<<<(L + 127) / 128, 128, 0, c->stream>>>(a, p, sc[P_BEAMS].as<double>());
  }
  KLU_TRY(check_launch("k_pa_cut"));
  {
    KLU_LAUNCH(c, "k_pa_rank");
    k_pa_rank<<<dim3(L, tiles), 256, 0, c->stream>>>(a, p);
  }
  KLU_TRY(check_launch("k_pa_rank"));
  {
    KLU_LAUNCH(c, "k_pa_connect");
    k_pa_connect<<<(int)(((int64_t)L * 32 + 127) / 128), 128, 0, c->stream>>>(a, p);
  }
  KLU_TRY(check_launch("k_pa_connect"));
  {
    KLU_LAUNCH(c, "k_prune_scan");
    k_prune_scan<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_scan"));
  KLU_TRY(scan_counts(c, a.arc_cnt, 0, L, c->d_res[5].as<int64_t>(), "k_scan_counts"));
  {
    KLU_LAUNCH(c, "k_pa_emit");
    k_pa_emit<<<dim3(L, tiles), 256, 0, c->stream>>>(a, p);
  }
  KLU_TRY(check_launch("k_pa_emit"));
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // seg_cnt is a stack object
  c->last_entries = -1;
  return 0;
}

int run_prune_dyn_beam(klu_ctx* c, const klu_opts* o) {
  if (!(o->beam_ratio > 0.0f && o->beam_ratio < 1.0f)) {
    set_error("--beam_ratio must be in the open range (0.0, 1.0).");  // :139-141
    return 1;
  }
  const int32_t L = c->L;
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = 0;
  CostParams cp = make_cost_params(o, false);
  KLU_TRY(run_tropical_sweeps(c, cp));
  if (L == 0) return 0;
  const int64_t S = std::max<int64_t>(c->S, 1), E = std::max<int64_t>(c->E, 1);
  enum { P_FB = 0, P_SMIN, P_FFB, P_BEAMS, P_CUT, P_ITERS, P_STATUS, P_AKEEP, P_SKEEP, P_ACNT, P_SCNT };
  KLU_TRY(c->d_scratch[P_FB].reserve(8 * E));
  KLU_TRY(c->d_scratch[P_SMIN].reserve(8 * S));
  KLU_TRY(c->d_scratch[P_FFB].reserve(8 * S));
  KLU_TRY(c->d_scratch[P_BEAMS].reserve(16 * (size_t)L));
  KLU_TRY(c->d_scratch[P_CUT].reserve(8 * (size_t)L));
  KLU_TRY(c->d_scratch[P_ITERS].reserve(4 * (size_t)L));
  KLU_TRY(c->d_scratch[P_STATUS].reserve(4 * (size_t)L));
  KLU_TRY(c->d_scratch[P_AKEEP].reserve(4 * E));
  KLU_TRY(c->d_scratch[P_SKEEP].reserve(4 * S));
  KLU_TRY(c->d_scratch[P_ACNT].reserve(4 * (size_t)L));
  KLU_TRY(c->d_scratch[P_SCNT].reserve(4 * (size_t)L));
  KLU_TRY(c->d_res[5].reserve(8 * (size_t)(L + 1)));
  for (int i = 0; i < 3; ++i) KLU_TRY(c->d_res[i].reserve(4 * E));
  KLU_TRY(c->d_res[3].reserve(4 * E));  // graph
  KLU_TRY(c->d_res[4].reserve(8 * E));  // acoustic (float) in the first half
  KLU_TRY(c->d_res[6].reserve(8 * S));  // state map (int32) | unused
  KLU_TRY(c->d_res[7].reserve(8 * S));  // fin_g | fin_a (float each)
  PruneArgs a;
  a.b = c->view();
  a.cp = cp;
  a.vfwd = c->d_vfwd.as<double>();
  a.vbwd = c->d_vbwd.as<double>();
  a.best = c->d_best.as<double>();
  a.fb = c->d_scratch[P_FB].as<double>();
  a.smin = c->d_scratch[P_SMIN].as<double>();
  a.ffb = c->d_scratch[P_FFB].as<double>();
  a.beam_ratio = o->beam_ratio;
  a.min_beam = o->min_beam;
  a.max_arcs = o->max_arcs;
  a.max_states = o->max_states;
  a.beams = c->d_scratch[P_BEAMS].as<double>();
  a.cutoff = c->d_scratch[P_CUT].as<double>();
  a.iters = c->d_scratch[P_ITERS].as<int>();
  a.status = c->d_scratch[P_STATUS].as<int>();
  a.arc_keep = c->d_scratch[P_AKEEP].as<int>();
  a.state_keep = c->d_scratch[P_SKEEP].as<int>();
  a.arc_cnt = c->d_scratch[P_ACNT].as<int>();
  a.state_cnt = c->d_scratch[P_SCNT].as<int>();
  a.res_off = c->d_res[5].as<int64_t>();
  a.o_arc = c->d_res[0].as<int32_t>();
  a.o_src = c->d_res[1].as<int32_t>();
  a.o_dst = c->d_res[2].as<int32_t>();
  a.o_g = c->d_res[3].as<float>();
  a.o_a = c->d_res[4].as<float>();
  a.o_smap = c->d_res[6].as<int32_t>();
  a.o_fg = c->d_res[7].as<float>();
  a.o_fa = c->d_res[7].as<float>() + S;
  a.inv_gs = 1.0 / (double)o->graph_scale;    // LatticeScale(1.0 / graph_scale, 1.0 / acoustic_scale), :145
  a.inv_as = 1.0 / (double)o->acoustic_scale;
  const int gs = c->num_sms * 8;
  {
    KLU_LAUNCH(c, "k_prune_fb");
    k_prune_fb<<<gs, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_fb"));
  {
    KLU_LAUNCH(c, "k_prune_smin");
    k_prune_smin<<<gs, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_smin"));
  {
    KLU_LAUNCH(c, "k_prune_search");
    k_prune_search<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_search"));
  int64_t max_arcs = 0;
  for (int32_t l = 0; l < L; ++l) max_arcs = std::max(max_arcs, c->h_e_off[l + 1] - c->h_e_off[l]);
  const int tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  {
    KLU_LAUNCH(c, "k_prune_mark");
    k_prune_mark<<<dim3(L, tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_mark"));
  {
    KLU_LAUNCH(c, "k_prune_scan");
    k_prune_scan<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_scan"));
  KLU_TRY(scan_counts(c, a.arc_cnt, 0, L, c->d_res[5].as<int64_t>(), "k_scan_counts"));
  {
    KLU_LAUNCH(c, "k_prune_emit");
    k_prune_emit<<<dim3(L, tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_prune_emit"));
  // a lattice whose loop cannot terminate is an error (the reference hangs on it)
  std::vector<int> status(L);
  KLU_CUDA(cudaMemcpyAsync(status.data(), a.status, 4 * (size_t)L, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  for (int32_t l = 0; l < L; ++l)
    if (status[l]) {
      set_error("lattice " + std::to_string(l) +
                ": infinite lattice beam (unreachable arcs); the reference's pruning loop does not terminate");
      return 1;
    }
  c->last_entries = -1;
  return 0;
}

}  // namespace klu

using namespace klu;

extern "C" int klu_fetch_prune(klu_ctx* c, int32_t* arc_index, int32_t* new_src, int32_t* new_dst, float* graph,
                               float* acoustic, int32_t* state_map, float* fin_graph, float* fin_acoustic,
                               double* beams) {
  if (c->last_tool != KLU_PRUNE_DYN_BEAM && c->last_tool != KLU_PRUNE_ARCS) {
    set_error("klu_fetch_prune: last run was not KLU_PRUNE_DYN_BEAM / KLU_PRUNE_ARCS");
    return 1;
  }
  KLU_CUDA(cudaSetDevice(c->device));
  if (c->last_entries < 0) {
    c->h_res_off.resize(c->L + 1);
    KLU_CUDA(cudaMemcpyAsync(c->h_res_off.data(), c->d_res[5].p, sizeof(int64_t) * (c->L + 1),
                             cudaMemcpyDeviceToHost, c->stream));
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    c->last_entries = c->h_res_off[c->L];
  }
  const size_t n = (size_t)c->last_entries, S = (size_t)c->S;
  auto get = [&](void* dst, const void* src, size_t bytes) -> int {
    if (dst && bytes) KLU_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    return 0;
  };
  KLU_TRY(get(arc_index, c->d_res[0].p, n * 4));
  KLU_TRY(get(new_src, c->d_res[1].p, n * 4));
  KLU_TRY(get(new_dst, c->d_res[2].p, n * 4));
  KLU_TRY(get(graph, c->d_res[3].p, n * 4));
  KLU_TRY(get(acoustic, c->d_res[4].p, n * 4));
  KLU_TRY(get(state_map, c->d_res[6].p, S * 4));
  KLU_TRY(get(fin_graph, c->d_res[7].p, S * 4));
  KLU_TRY(get(fin_acoustic, c->d_res[7].as<float>() + std::max<size_t>(S, 1), S * 4));
  KLU_TRY(get(beams, c->d_scratch[3].p, 16 * (size_t)c->L));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}
