// klu_bestpath.cu -- decode stage of lattice-best-path2 (SURVEY.md K11).
//
// Reference: latbin/lattice-best-path2.cc:149-199.  After the (label, position)
// posteriors, the reference builds a tropical FST over the length-unfolded lattice
// (fstext/fstext-utils2.h:109-215) padded with a chain of kNoLabel arcs
// (fstext/fstext-utils2.h:218-271), arc cost (float) 1 - P(label, position), and
// takes fst::ShortestPath(n = 1) [ext].  Nothing is materialised here:
//   * a banded float min-plus sweep over (state, #labels) cells, pulling over the
//     incoming arcs of the packed lattice, with parent pointers;
//   * ties are broken the way OpenFst's single-source shortest path on a
//     top-sorted FST does: the parent is the first relaxing arc, in increasing
//     (unfolded source id, arc position) order, that reaches the final minimum;
//     the unfolded id is the rank of (length, input state id), arc position is the
//     order after ArcSort(olabel) (:107);
//   * the padding chain aux[k] is a short serial scan per lattice;
//   * a backtrace emits the labels (epsilon and kNoLabel stripped, :195-199).
#include <math.h>

#include <algorithm>

#include "klu_common.cuh"

namespace klu {

namespace {

struct BpArgs {
  BatchView b;
  CostParams cp;
  int l0, l1;
  long long band_base;
  const double* alpha2;
  const double* beta;
  const long long* arc_cellbase;
  const double* ecost;
  float* d2;       // chunk-local cells
  int32_t* par;    // chunk-local cells: in-order arc (global index) or -1
  const int32_t* maxlen;   // [L]
  const int64_t* pad_off;  // [L+1] offsets of the per-lattice chain arrays (maxlen+2 each)
  float* padcost;          // cost of aux[k-1] -> aux[k] at [pad_off + k]
  double* fscratch;        // [pad_off ...] F_k then fw[aux_k]
  const int64_t* lab_off;  // [L+1] label regions (capacity maxlen each)
  int32_t* labels;
  int32_t* lab_cnt;        // [L]
  float* cost;             // [L]
  int* counter;
};

struct Cand {
  float v;
  unsigned long long k1, k2;  // (len_u, input id of u), (label, input arc index)
  int e;
};

__device__ __forceinline__ bool cand_less(const Cand& a, const Cand& b) {
  if (a.v != b.v) return a.v < b.v;
  if (a.k1 != b.k1) return a.k1 < b.k1;
  return a.k2 < b.k2;
}

// (state, len) min-plus sweep.  One CTA owns one lattice (work queue); a level's cells are
// spread over the threads with consecutive threads on consecutive lengths, and the level's
// incoming arcs are staged once per piece in shared memory (where the source's band starts
// on the length axis, its valid range, where the arc's (label, position) costs start, the
// two tie-break keys), exactly as k_banded_alpha does for the log semiring: the cost and the
// predecessor's distance are then contiguous reads along the length axis.
constexpr int kBpThreads = 512;
constexpr int kBpArcs = 512;
constexpr int kBpStates = 128;

__global__ void __launch_bounds__(kBpThreads) k_bp_viterbi(BpArgs a) {
  __shared__ long long sv_base[kBpArcs];   // d2 index of (source, len - nz) = base + len
  __shared__ long long sv_cost[kBpArcs];   // cost index of (arc, len - nz) = cost + len; LLONG_MIN: epsilon arc
  __shared__ unsigned long long sv_k2[kBpArcs];  // (label, input arc index)
  __shared__ int2 sv_range[kBpArcs];       // valid len: [x, y)
  __shared__ int2 sv_src[kBpArcs];         // (input id of the source, nz)
  __shared__ int ss_arc[kBpStates + 1];
  __shared__ long long ss_cell[kBpStates + 1];
  __shared__ int ss_lo[kBpStates];
  __shared__ int s_item, s_take;
  const BatchView& b = a.b;
  float* d2 = a.d2 - a.band_base;
  int32_t* par = a.par - a.band_base;
  const float inf = __int_as_float(0x7f800000);
  const long long kEps = (long long)0x8000000000000000LL;
  const int tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) s_item = atomicAdd(a.counter, 1);
    __syncthreads();
    if (s_item >= a.l1 - a.l0) break;
    const int l = a.l0 + s_item;
    const int s_begin = b.s_off[l], s_end = b.s_off[l + 1];
    if (s_begin == s_end) continue;
    const int* lv = b.lvl_start + b.lvl_off[l];
    const int nl = b.lvl_off[l + 1] - b.lvl_off[l] - 1;
    for (int s = lv[0] + tid; s < lv[1]; s += kBpThreads)
      if (s == s_begin && b.band_off[s + 1] > b.band_off[s]) {
        d2[b.band_off[s]] = 0.0f;
        par[b.band_off[s]] = -1;
      }
    for (int j = 1; j < nl; ++j) {
      const int a1 = lv[j + 1];
      int s0 = lv[j];
      while (s0 < a1) {
        __syncthreads();
        const int nst = min(a1 - s0, kBpStates);
        for (int k = tid; k <= nst; k += kBpThreads) {
          ss_arc[k] = b.in_off[s0 + k];
          ss_cell[k] = b.band_off[s0 + k];
          if (k < nst) ss_lo[k] = b.band_lo[s0 + k];
        }
        if (tid == 0) s_take = 1;
        __syncthreads();
        const int e_base = ss_arc[0];
        for (int k = tid + 1; k <= nst; k += kBpThreads)
          if (ss_arc[k] - e_base <= kBpArcs) atomicMax(&s_take, k);
        __syncthreads();
        const int take = s_take;
        const int narcs = ss_arc[take] - e_base;
        const bool staged = narcs <= kBpArcs;  // else: one state with more arcs than fit (take == 1)
        if (staged) {
          for (int i = tid; i < narcs; i += kBpThreads) {
            const int4 r = __ldg(b.in_rec + e_base + i);
            const int plo = b.band_lo[r.x];
            const int pw = (int)(b.band_off[r.x + 1] - b.band_off[r.x]);
            const int nz = r.w != 0 ? 1 : 0;
            const int eo = b.in2out[e_base + i];
            sv_base[i] = b.band_off[r.x] - plo - nz;
            sv_range[i] = (plo < 0 || pw <= 0) ? make_int2(0, 0) : make_int2(plo + nz, plo + pw + nz);
            sv_cost[i] = nz ? a.arc_cellbase[eo] - nz : kEps;
            sv_src[i] = make_int2(b.orig[r.x], nz);
            sv_k2[i] = ((unsigned long long)(unsigned int)r.w << 32) | (unsigned int)b.out_orig[eo];
          }
        }
        __syncthreads();
        const long long c0 = ss_cell[0], c1 = ss_cell[take];
        for (long long cell = c0 + tid; cell < c1; cell += kBpThreads) {
          const int lo = last_le(ss_cell, 0, take - 1, cell);  // last k with ss_cell[k] <= cell
          const int len = ss_lo[lo] + (int)(cell - ss_cell[lo]);
          Cand best;
          best.v = inf;
          best.k1 = ~0ULL;
          best.k2 = ~0ULL;
          best.e = -1;
          if (staged) {
            const int i1 = ss_arc[lo + 1] - e_base;
#pragma unroll 2
            for (int i = ss_arc[lo] - e_base; i < i1; ++i) {
              const int2 rg = sv_range[i];
              if (len < rg.x || len >= rg.y) continue;
              const float du = d2[sv_base[i] + len];
              if (!(du < inf)) continue;
              const long long cb = sv_cost[i];
              const float w = cb == kEps ? 0.0f : (float)a.ecost[cb + len];
              const int2 sn = sv_src[i];
              Cand cnd;
              cnd.v = __fadd_rn(du, w);
              cnd.k1 = ((unsigned long long)(unsigned int)(len - sn.y) << 32) | (unsigned int)sn.x;
              cnd.k2 = sv_k2[i];
              cnd.e = e_base + i;
              if (cand_less(cnd, best)) best = cnd;
            }
          } else {
            const int s = s0 + lo;
            for (int e = b.in_off[s]; e < b.in_off[s + 1]; ++e) {
              const int4 r = __ldg(b.in_rec + e);
              const int nz = r.w != 0 ? 1 : 0;
              const int plen = len - nz;
              const int plo = b.band_lo[r.x];
              const int pw = (int)(b.band_off[r.x + 1] - b.band_off[r.x]);
              if (plo < 0 || plen < plo || plen >= plo + pw) continue;
              const float du = d2[b.band_off[r.x] + plen - plo];
              if (!(du < inf)) continue;
              const int eo = b.in2out[e];
              float w = 0.0f;
              if (nz) w = (float)a.ecost[a.arc_cellbase[eo] + plen];
              Cand cnd;
              cnd.v = __fadd_rn(du, w);
              cnd.k1 = ((unsigned long long)(unsigned int)plen << 32) | (unsigned int)b.orig[r.x];
              cnd.k2 = ((unsigned long long)(unsigned int)r.w << 32) | (unsigned int)b.out_orig[eo];
              cnd.e = e;
              if (cand_less(cnd, best)) best = cnd;
            }
          }
          d2[cell] = best.v;
          par[cell] = best.e;
        }
        s0 += take;
      }
    }
  }
}

// One warp per lattice: costs of the padding arcs.  fw[aux_k] folds, in the
// unfolded state order, the final states with k labels, then the chain arc.
__global__ void __launch_bounds__(128) k_bp_pad(BpArgs a) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= a.l1 - a.l0) return;
  const int l = a.l0 + warp;
  const BatchView& b = a.b;
  const int s0 = b.s_off[l], s1 = b.s_off[l + 1];
  if (s0 == s1) return;
  const int maxlen = a.maxlen[l];
  double* F = a.fscratch + a.pad_off[l];
  float* pc = a.padcost + a.pad_off[l];
  const double* alpha2 = a.alpha2 - a.band_base;
  for (int k = lane; k <= maxlen; k += 32) F[k] = neg_inf();
  __syncwarp();
  // the reference folds the final states in unfolded-id order; here in packed
  // order, which only perturbs the last ulp of each LogAdd
  for (int s = s0; s < s1; ++s) {
    const float fg = b.fin_g[s], fa = b.fin_a[s];
    if (isinf(fg) && isinf(fa)) continue;
    const int lo = b.band_lo[s];
    if (lo < 0) continue;
    const int w = (int)(b.band_off[s + 1] - b.band_off[s]);
    const double fc = final_cost(fg, fa, a.cp);
    for (int i = lane; i < w; i += 32) F[lo + i] = log_add(F[lo + i], alpha2[b.band_off[s] + i] - fc);
    __syncwarp();
  }
  if (lane == 0) {
    const double norm = a.beta[s0];
    double fw = neg_inf();
    pc[0] = 0.0f;
    for (int k = 0; k < maxlen; ++k) {
      fw = log_add(fw, F[k]);
      const double post = fmin(0.0, fw - norm);
      double ls;
      if (post >= 0.0) ls = neg_inf();
      else {
        ls = log(1.0 - exp(post));
        if (ls != ls) ls = neg_inf();
      }
      pc[k + 1] = (float)exp(ls);  // arc aux[k] -> aux[k+1], key (kNoLabel, k+1)
    }
  }
}

// One thread per lattice: chain aux[0..maxlen], final selection, backtrace.
__global__ void __launch_bounds__(128) k_bp_trace(BpArgs a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.l1 - a.l0) return;
  const int l = a.l0 + t;
  const BatchView& b = a.b;
  const int s0 = b.s_off[l], s1 = b.s_off[l + 1];
  const float inf = __int_as_float(0x7f800000);
  if (s0 == s1) {
    a.lab_cnt[l] = 0;
    a.cost[l] = inf;
    return;
  }
  const float* d2 = a.d2 - a.band_base;
  const int32_t* par = a.par - a.band_base;
  const int maxlen = a.maxlen[l];
  const float* pc = a.padcost + a.pad_off[l];
  // per length: best final (value, then smaller input id), kept in the F scratch
  // as two int32 (state, bits of value)
  int2* bf = reinterpret_cast<int2*>(a.fscratch + a.pad_off[l]);
  for (int k = 0; k <= maxlen; ++k) bf[k] = make_int2(-1, __float_as_int(inf));
  for (int s = s0; s < s1; ++s) {
    const float fg = b.fin_g[s], fa = b.fin_a[s];
    if (isinf(fg) && isinf(fa)) continue;
    const int lo = b.band_lo[s];
    if (lo < 0) continue;
    const int w = (int)(b.band_off[s + 1] - b.band_off[s]);
    for (int i = 0; i < w; ++i) {
      const float v = __fadd_rn(d2[b.band_off[s] + i], 0.0f);
      if (!(v < inf)) continue;
      const int2 cur = bf[lo + i];
      const float cv = __int_as_float(cur.y);
      if (v < cv || (v == cv && (cur.x < 0 || b.orig[s] < b.orig[cur.x]))) bf[lo + i] = make_int2(s, __float_as_int(v));
    }
  }
  // chain: d[aux_k] = min(best final of length k, d[aux_{k-1}] + pad_k), strict improvement for the chain
  float d = inf;
  int from_final_k = -1;  // the k at which the winning path entered the chain
  for (int k = 0; k <= maxlen; ++k) {
    float viaf = __int_as_float(bf[k].y);
    float dk = viaf;
    int src_k = viaf < inf ? k : -1;
    if (k > 0 && d < inf) {
      const float via_chain = __fadd_rn(d, pc[k]);
      if (via_chain < dk) {
        dk = via_chain;
        src_k = from_final_k;
      }
    }
    d = dk;
    from_final_k = src_k;
  }
  a.cost[l] = __fadd_rn(d, 0.0f);
  int32_t* out = a.labels + a.lab_off[l];
  int n = 0;
  if (d < inf && from_final_k >= 0) {
    int s = bf[from_final_k].x;
    int len = from_final_k;
    // walk back to the start, labels come out reversed
    while (true) {
      const int e = par[b.band_off[s] + (len - b.band_lo[s])];
      if (e < 0) break;
      const int4 r = b.in_rec[e];
      if (r.w != 0) {
        out[n++] = r.w;
        len -= 1;
      }
      s = r.x;
    }
    for (int i = 0; i < n / 2; ++i) {
      const int32_t tmp = out[i];
      out[i] = out[n - 1 - i];
      out[n - 1 - i] = tmp;
    }
  }
  a.lab_cnt[l] = n;
}

__global__ void __launch_bounds__(128) k_bp_compact(const int64_t* lab_off, const int32_t* labels, const int32_t* cnt,
                                                    const int64_t* res_off, int32_t* dense, int L) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= L) return;
  const int n = cnt[warp];
  for (int i = lane; i < n; i += 32) dense[res_off[warp] + i] = labels[lab_off[warp] + i];
}

}  // namespace

// scratch slots owned by best-path2 (distinct from the index pipeline's 0..11)
int best_path2_decode(klu_ctx* c, const CostParams& cp, const BestPathChunk& ch) {
  const int32_t L = c->L;
  // per-batch layout of the chain / label regions, built on the first chunk
  DevBuf& d_maxlen = c->d_res[0];
  DevBuf& d_padoff = c->d_res[1];
  DevBuf& d_laboff = c->d_res[2];
  DevBuf& d_labels = c->d_res[3];
  DevBuf& d_labcnt = c->d_res[6];
  DevBuf& d_cost = c->d_res[7];
  std::vector<int64_t> pad_off(L + 1, 0), lab_off(L + 1, 0);
  for (int32_t l = 0; l < L; ++l) {
    pad_off[l + 1] = pad_off[l] + c->h_maxlen[l] + 2;
    lab_off[l + 1] = lab_off[l] + c->h_maxlen[l];
  }
  if (ch.first_chunk) {
    KLU_TRY(d_maxlen.reserve(4 * (size_t)L));
    KLU_TRY(d_padoff.reserve(8 * (size_t)(L + 1)));
    KLU_TRY(d_laboff.reserve(8 * (size_t)(L + 1)));
    KLU_TRY(d_labels.reserve(4 * (size_t)std::max<int64_t>(lab_off[L], 1)));
    KLU_TRY(d_labcnt.reserve(4 * (size_t)L));
    KLU_TRY(d_cost.reserve(4 * (size_t)L));
    KLU_CUDA(cudaMemcpyAsync(d_maxlen.p, c->h_maxlen.data(), 4 * (size_t)L, cudaMemcpyHostToDevice, c->stream));
    KLU_CUDA(cudaMemcpyAsync(d_padoff.p, pad_off.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
    KLU_CUDA(cudaMemcpyAsync(d_laboff.p, lab_off.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
    KLU_CUDA(cudaStreamSynchronize(c->stream));
  }
  const long long cells = c->h_band_off[ch.l1] - ch.band_base;
  // Viterbi cells and chain scratch live in the otherwise idle tropical buffers
  KLU_TRY(c->d_vfwd.reserve(4 * (size_t)std::max<long long>(cells, 1)));
  KLU_TRY(c->d_vbwd.reserve(4 * (size_t)std::max<long long>(cells, 1)));
  KLU_TRY(c->d_best.reserve(8 * (size_t)pad_off[L] + 8));
  KLU_TRY(c->d_totfwd.reserve(4 * (size_t)pad_off[L] + 8));
  BpArgs a;
  a.b = c->view();
  a.cp = cp;
  a.l0 = ch.l0;
  a.l1 = ch.l1;
  a.band_base = ch.band_base;
  a.alpha2 = ch.alpha2;
  a.beta = c->d_beta.as<double>();
  a.arc_cellbase = ch.arc_cellbase;
  a.ecost = ch.ecost;
  a.d2 = c->d_vfwd.as<float>();
  a.par = c->d_vbwd.as<int32_t>();
  a.maxlen = d_maxlen.as<int32_t>();
  a.pad_off = d_padoff.as<int64_t>();
  a.padcost = c->d_totfwd.as<float>();
  a.fscratch = c->d_best.as<double>();
  a.lab_off = d_laboff.as<int64_t>();
  a.labels = d_labels.as<int32_t>();
  a.lab_cnt = d_labcnt.as<int32_t>();
  a.cost = d_cost.as<float>();
  KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));
  a.counter = c->d_counter.as<int>();
  const int nl = ch.l1 - ch.l0;
  // every cell of the chunk is written by the sweep (unreachable ones as +inf, parent -1)
  {
    KLU_LAUNCH(c, "k_bp_pad");
    k_bp_pad<<<(nl * 32 + 127) / 128, 128, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_bp_pad"));
  {
    KLU_LAUNCH(c, "k_bp_viterbi");
    const int grid = std::max(1, std::min(nl, c->num_sms * 8));  // one CTA per lattice in flight
    k_bp_viterbi<<<grid, kBpThreads, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_bp_viterbi"));
  {
    KLU_LAUNCH(c, "k_bp_trace");
    k_bp_trace<<<(nl + 127) / 128, 128, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_bp_trace"));
  if (ch.l1 == L) {  // last chunk: dense label table
    KLU_TRY(c->d_res[5].reserve(8 * (size_t)(L + 1)));
    KLU_TRY(c->d_res[4].reserve(4 * (size_t)std::max<int64_t>(lab_off[L], 1)));
    KLU_TRY(scan_counts(c, a.lab_cnt, 0, L, c->d_res[5].as<int64_t>(), "k_scan_counts"));
    {
      KLU_LAUNCH(c, "k_bp_compact");
      k_bp_compact<<<(L * 32 + 127) / 128, 128, 0, c->stream>>>(a.lab_off, a.labels, a.lab_cnt,
                                                                 c->d_res[5].as<int64_t>(), c->d_res[4].as<int32_t>(), L);
    }
    KLU_TRY(check_launch("k_bp_compact"));
  }
  return 0;
}

}  // namespace klu

using namespace klu;

extern "C" int klu_fetch_best_path2(klu_ctx* c, int32_t* label, float* cost, int32_t* num_frames) {
  if (c->last_tool != KLU_BEST_PATH2) {
    set_error("klu_fetch_best_path2: last run was not KLU_BEST_PATH2");
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
  const size_t n = (size_t)c->last_entries;
  if (label && n) KLU_CUDA(cudaMemcpyAsync(label, c->d_res[4].p, n * 4, cudaMemcpyDeviceToHost, c->stream));
  if (cost && c->L) KLU_CUDA(cudaMemcpyAsync(cost, c->d_res[7].p, 4 * (size_t)c->L, cudaMemcpyDeviceToHost, c->stream));
  if (num_frames) memcpy(num_frames, c->h_num_frames.data(), sizeof(int32_t) * c->L);
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}
