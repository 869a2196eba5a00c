// klu_gpack.cu -- GPU lattice packer (north_star subsystem 1, SURVEY.md K0).
//
// Same output as the host packer in klu_pack.cu (level-bucketed states, arc
// records in source and destination order, CSR offsets, times, length bands,
// frame -> arc CSR) but built on the device: the caller's SoA arrays go H2D as
// they are (asynchronous when they live in klu_host_alloc memory) and every
// restructuring step runs at HBM speed instead of on the host cores:
//   1. per-state first-arc offsets (binary search in the src-sorted arc list) and
//      validation of the layout contract;
//   2. one warp per lattice walks the states in topological (= input) order and
//      pushes level / frame time / label-count band along the outgoing arcs
//      (integer atomics: order independent, hence deterministic);
//   3. states are stable-sorted by level with the segmented radix sort;
//   4. arcs are scattered to source order (state blocks move as a whole, no sort)
//      and stable-sorted by destination for the pull order of the forward sweep;
//   5. per-lattice scans build the CSR offsets, the band offsets and the
//      frame -> arc CSR.
// Two small D2H copies (per-lattice metadata) are the only host round trips.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <numeric>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

enum { M_NL = 0, M_FRAMES, M_TIMES_OK, M_MAXLEN, M_MAXLABEL, M_MAXTIME, M_ERR, M_PAD, M_STRIDE };

struct GP {
  int L, S, E;
  const int64_t *s_off64, *e_off64;
  const int32_t *s_off, *e_off;
  const int32_t *src, *dst, *label, *dur, *fdur;
  const float *g, *a, *fg, *fa;
  int32_t* first_arc;  // [S+1] by input state (global)
  int32_t* level;      // [S] by input state
  int32_t* time;       // [S] by input state
  int32_t *blo, *bhi;  // [S] by input state
  int32_t* meta;       // [L * M_STRIDE]
  long long* cap;      // [L * 2]: arc x frame instances, arc x length instances
  // packed outputs
  int32_t* old2new;    // [S] input state (global) -> packed state (global)
  int32_t *orig, *plevel, *ptime, *band_lo, *lvl_start, *in_off, *out_off, *out_src, *out_orig, *in2out;
  const int32_t *lvl_off, *fr_base;
  float *pfg, *pfa;
  int64_t *band_off, *fr_off;
  int4 *in_rec, *out_rec;
  int32_t* frame_arc;
  int32_t* counts;     // [S] scratch: per packed state count to be scanned
  int32_t* fr_cnt;     // per frame slot
  long long* lat_tot;  // [L+1] per-lattice totals / bases
};

__device__ __forceinline__ int ld_cg_i32(const int32_t* p) { return __ldcg(p); }

// grid (L, tiles): first arc of every state + layout validation
__global__ void __launch_bounds__(256) k_gp_first_arc(GP a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
  const int e0 = a.e_off[l], e1 = a.e_off[l + 1];
  const int t = lt.tile * blockDim.x + threadIdx.x, stride = lt.tiles * blockDim.x;
  for (int s = t; s < ns; s += stride) {
    int lo = e0, hi = e1;  // first arc with src >= s
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (a.src[mid] < s) lo = mid + 1;
      else hi = mid;
    }
    a.first_arc[s0 + s] = lo;
  }
  if (l == a.L - 1 && t == 0) a.first_arc[a.S] = a.E;
  int bad = 0;
  for (int e = e0 + t; e < e1; e += stride) {
    const int u = a.src[e], v = a.dst[e];
    if (u < 0 || u >= ns || v <= u || v >= ns) bad = 1;
    if (e > e0 && a.src[e - 1] > u) bad = 1;
    if (!isfinite(a.g[e]) || !isfinite(a.a[e])) bad = 2;
  }
  if (bad) atomicMax(&a.meta[l * M_STRIDE + M_ERR], bad);
}

// grid (L, tiles): source state of every arc from the per-state first-arc offsets (input
// without arc_src)
__global__ void __launch_bounds__(256) k_gp_expand_src(GP a, int32_t* src_out) {
  const int l = blockIdx.x;
  const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
  const int e_end = a.e_off[l + 1];
  for (int s = blockIdx.y * blockDim.x + threadIdx.x; s < ns; s += gridDim.y * blockDim.x) {
    const int f0 = a.first_arc[s0 + s];
    const int f1 = s + 1 < ns ? a.first_arc[s0 + s + 1] : e_end;
    for (int e = f0; e < f1; ++e) src_out[e] = s;
  }
}

// compact input forms -> the 32-bit arrays the packer works on (klu_lattices.arc_dur_u8 / arc_dst_delta_u16)
__global__ void __launch_bounds__(256) k_gp_expand_compact(const uint8_t* dur8, const uint16_t* delta16, const uint16_t* label16,
                                                           const int32_t* src, int32_t* dur, int32_t* dst, int32_t* label,
                                                           int64_t E) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
    if (dur8) dur[e] = (int32_t)dur8[e];
    if (delta16) dst[e] = src[e] + (int32_t)delta16[e];
    if (label16) label[e] = (int32_t)label16[e];
  }
}

// one warp per lattice: levels, state times, label-count bands, per-lattice stats
__global__ void __launch_bounds__(128) k_gp_levels(GP a, int* counter) {
  const int lane = threadIdx.x & 31;
  for (;;) {
    int l = 0;
    if (lane == 0) l = atomicAdd(counter, 1);
    l = __shfl_sync(0xffffffffu, l, 0);
    if (l >= a.L) break;
    const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
    int32_t* meta = a.meta + l * M_STRIDE;
    if (ns == 0 || meta[M_ERR] != 0) {
      if (lane == 0) {
        meta[M_NL] = 0;
        meta[M_FRAMES] = 0;
        meta[M_TIMES_OK] = 1;
        meta[M_MAXLEN] = 0;
        meta[M_MAXLABEL] = 0;
        meta[M_MAXTIME] = 0;
      }
      continue;
    }
    for (int s = lane; s < ns; s += 32) {
      a.level[s0 + s] = 0;
      a.time[s0 + s] = s == 0 ? 0 : -1;
      a.blo[s0 + s] = s == 0 ? 0 : 0x7fffffff;
      a.bhi[s0 + s] = s == 0 ? 0 : -1;
    }
    __threadfence();
    __syncwarp();
    int times_ok = 1, max_label = 0;
    // The arcs of a state do not depend on what the walk computes: the first 32 of the NEXT state
    // (and its arc range) are fetched before the current state's values are waited for, so only
    // the level / time / band loads stay on the chain of ns dependent steps.
    int f0 = a.first_arc[s0], f1 = a.first_arc[s0 + 1];
    int pd = 0, pl = 0, pu = 0;
    if (f0 + lane < f1) {
      pd = a.dst[f0 + lane];
      pl = a.label[f0 + lane];
      pu = a.dur[f0 + lane];
    }
    for (int s = 0; s < ns; ++s) {
      const int gs = s0 + s;
      const int nf0 = f1, nf1 = s + 1 < ns ? a.first_arc[gs + 2] : f1;
      int nd = 0, nlb = 0, nu = 0;
      if (nf0 + lane < nf1) {
        nd = a.dst[nf0 + lane];
        nlb = a.label[nf0 + lane];
        nu = a.dur[nf0 + lane];
      }
      const int lev = ld_cg_i32(a.level + gs), ts = ld_cg_i32(a.time + gs);
      const int lo = ld_cg_i32(a.blo + gs), hi = ld_cg_i32(a.bhi + gs);
      for (int e = f0 + lane; e < f1; e += 32) {
        const bool first = e < f0 + 32;
        const int d = s0 + (first ? pd : a.dst[e]);
        const int lab = first ? pl : a.label[e];
        const int du = first ? pu : a.dur[e];
        atomicMax(a.level + d, lev + 1);
        if (ts >= 0) {
          const int tv = ts + du;
          const int old = atomicCAS(a.time + d, -1, tv);
          if (old != -1 && old != tv) times_ok = 0;
        }
        if (hi >= 0) {
          const int nz = lab != 0 ? 1 : 0;
          atomicMin(a.blo + d, lo + nz);
          atomicMax(a.bhi + d, hi + nz);
        }
        max_label = max(max_label, lab);
      }
      __threadfence();
      __syncwarp();
      f0 = nf0;
      f1 = nf1;
      pd = nd;
      pl = nlb;
      pu = nu;
    }
    int nl = 0, frames = -1, maxlen = 0, maxtime = 0;
    for (int s = lane; s < ns; s += 32) {
      const int gs = s0 + s;
      nl = max(nl, ld_cg_i32(a.level + gs) + 1);
      const int ts = ld_cg_i32(a.time + gs);
      maxtime = max(maxtime, ts);
      maxlen = max(maxlen, ld_cg_i32(a.bhi + gs));
      const float fg = a.fg[gs], fa = a.fa[gs];
      if (!(isinf(fg) && isinf(fa)) && ts >= 0) frames = max(frames, ts + (a.fdur ? a.fdur[gs] : 0));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      nl = max(nl, __shfl_xor_sync(0xffffffffu, nl, o));
      frames = max(frames, __shfl_xor_sync(0xffffffffu, frames, o));
      maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
      maxtime = max(maxtime, __shfl_xor_sync(0xffffffffu, maxtime, o));
      max_label = max(max_label, __shfl_xor_sync(0xffffffffu, max_label, o));
      times_ok = min(times_ok, __shfl_xor_sync(0xffffffffu, times_ok, o));
    }
    if (lane == 0) {
      meta[M_NL] = nl;
      meta[M_FRAMES] = frames < 0 ? 0 : frames;
      meta[M_TIMES_OK] = times_ok;
      meta[M_MAXLEN] = maxlen;
      meta[M_MAXLABEL] = max_label;
      meta[M_MAXTIME] = max(maxtime, frames);
    }
  }
}

// sort keys of the states: (level, input id) -> stable sort on level
__global__ void __launch_bounds__(256) k_gp_state_keys(GP a, unsigned long long* key, unsigned int* val) {
  const int l = blockIdx.x;
  const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
  for (int s = blockIdx.y * blockDim.x + threadIdx.x; s < ns; s += gridDim.y * blockDim.x) {
    key[s0 + s] = (unsigned long long)(unsigned int)a.level[s0 + s];
    val[s0 + s] = (unsigned int)s;
  }
}

// per packed state: permutation, level starts, per-state payload, out-degree
__global__ void __launch_bounds__(256) k_gp_state_perm(GP a, const unsigned long long* key_a,
                                                        const unsigned long long* key_b, const unsigned int* val_a,
                                                        const unsigned int* val_b, const unsigned char* where) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
  const unsigned long long* key = (where[l] ? key_b : key_a) + s0;
  const unsigned int* val = (where[l] ? val_b : val_a) + s0;
  int32_t* lv = a.lvl_start + a.lvl_off[l];
  const int nl = a.lvl_off[l + 1] - a.lvl_off[l] - 1;
  for (int n = lt.tile * blockDim.x + threadIdx.x; n < ns; n += lt.tiles * blockDim.x) {
    const int old = (int)val[n];
    const int lev = (int)key[n];
    const int go = s0 + old, gn = s0 + n;
    a.old2new[go] = gn;
    a.orig[gn] = old;
    a.plevel[gn] = lev;
    a.ptime[gn] = a.time[go];
    a.pfg[gn] = a.fg[go];
    a.pfa[gn] = a.fa[go];
    const int hi = a.bhi[go];
    a.band_lo[gn] = hi >= 0 ? a.blo[go] : -1;
    a.counts[gn] = a.first_arc[go + 1] - a.first_arc[go];
    if (n == 0 || (int)key[n - 1] != lev) lv[lev] = gn;
    if (n == ns - 1) lv[nl] = s0 + ns;
  }
  if (ns == 0 && lt.tile == 0 && threadIdx.x == 0) lv[0] = s0;
}

// One CTA per lattice: exclusive scan of per-state int32 counts.  MODE 0: out32 =
// base32[l] + prefix; MODE 1: lattice-local prefix as int64 + lattice total.
template <int MODE>
__global__ void __launch_bounds__(256) k_gp_lat_scan(const int32_t* cnt, const int32_t* seg_off,
                                                     const int32_t* base32, int32_t* out32, int64_t* out64,
                                                     long long* lat_tot) {
  __shared__ long long warp_sum[8];
  __shared__ long long carry_s;
  const int l = blockIdx.x;
  const int i0 = seg_off[l], n = seg_off[l + 1] - i0;
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = 0; tile < n; tile += 256) {
    const int i = tile + tid;
    const long long c = i < n ? cnt[i0 + i] : 0;
    const long long pre = cta_exclusive_scan<long long, 256>(c, warp_sum, carry_s);
    if (i < n) {
      if (MODE == 0) out32[i0 + i] = base32[l] + (int32_t)(pre);
      else out64[i0 + i] = pre;
    }
  }
  if (tid == 0 && MODE == 1) lat_tot[l] = carry_s;
}

// lattice-local int64 offsets -> global: off[i] += base[l]; also the closing entry
__global__ void __launch_bounds__(256) k_gp_add_base(int64_t* off, const int32_t* seg_off, const long long* base,
                                                     int L, int64_t* closing) {
  const int l = blockIdx.x;
  const int i0 = seg_off[l], n = seg_off[l + 1] - i0;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i < n; i += gridDim.y * blockDim.x) off[i0 + i] += base[l];
  if (l == L - 1 && blockIdx.y == 0 && threadIdx.x == 0) *closing = base[L];
}

// grid (L, tiles): arcs to source order + per-lattice capacities of the expansions
__global__ void __launch_bounds__(256) k_gp_scatter(GP a, unsigned int* key, unsigned int* val) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  __shared__ long long red[2][8];
  const int l = lt.l;
  const int s0 = a.s_off[l];
  const int e0 = a.e_off[l], e1 = a.e_off[l + 1];
  const int T = a.meta[l * M_STRIDE + M_FRAMES];
  long long cf = 0, cp = 0;
  int span = 0;
  for (int e = e0 + lt.tile * blockDim.x + threadIdx.x; e < e1; e += lt.tiles * blockDim.x) {
    const int go = s0 + a.src[e], gd = s0 + a.dst[e];
    span = max(span, a.dur[e]);
    const int n = a.old2new[go], d = a.old2new[gd];
    const int p = a.out_off[n] + (e - a.first_arc[go]);
    const int lab = a.label[e];
    a.out_rec[p] = make_int4(d, __float_as_int(a.g[e]), __float_as_int(a.a[e]), lab);
    a.out_src[p] = n;
    a.out_orig[p] = e - e0;
    key[p] = (unsigned int)(d - s0);  // sort key of the in-order: local packed dst (32-bit keys)
    val[p] = (unsigned int)(p - e0);
    if (lab != 0) {
      const int fa = max(a.time[go], 0), fb = min(a.time[gd], T);
      cf += fb > fa ? fb - fa : 0;
      const int hi = a.bhi[go];
      cp += hi >= 0 ? hi - a.blo[go] + 1 : 0;
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cf += __shfl_xor_sync(0xffffffffu, cf, o);
    cp += __shfl_xor_sync(0xffffffffu, cp, o);
    span = max(span, __shfl_xor_sync(0xffffffffu, span, o));
  }
  if (lane == 0) {
    red[0][warp] = cf;
    red[1][warp] = cp;
    if (span > 0) atomicMax(&a.meta[a.L * M_STRIDE], span);  // spare meta row: longest arc of the batch
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    long long x = 0, y = 0;
    for (int w = 0; w < 8; ++w) {
      x += red[0][w];
      y += red[1][w];
    }
    if (x) atomicAdd(reinterpret_cast<unsigned long long*>(a.cap + 2 * l), (unsigned long long)x);
    if (y) atomicAdd(reinterpret_cast<unsigned long long*>(a.cap + 2 * l + 1), (unsigned long long)y);
  }
}

// grid (L, tiles): destination-ordered records from the sorted (dst, out position) pairs
__global__ void __launch_bounds__(256) k_gp_in_build(GP a, const unsigned int* key_a,
                                                     const unsigned int* key_b, const unsigned int* val_a,
                                                     const unsigned int* val_b, const unsigned char* where) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
  const int e0 = a.e_off[l], na = a.e_off[l + 1] - e0;
  const unsigned int* key = (where[l] ? key_b : key_a) + e0;
  const unsigned int* val = (where[l] ? val_b : val_a) + e0;
  const int t = lt.tile * blockDim.x + threadIdx.x, stride = lt.tiles * blockDim.x;
  for (int q = t; q < na; q += stride) {
    const int p = e0 + (int)val[q];
    const int4 r = a.out_rec[p];
    a.in_rec[e0 + q] = make_int4(a.out_src[p], r.y, r.z, r.w);
    a.in2out[e0 + q] = p;
  }
  for (int n = t; n < ns; n += stride) {
    int lo = 0, hi = na;  // first sorted arc with dst >= n
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if ((int)key[mid] < n) lo = mid + 1;
      else hi = mid;
    }
    a.in_off[s0 + n] = e0 + lo;
  }
  if (l == a.L - 1 && t == 0) {
    a.in_off[a.S] = a.E;
    a.out_off[a.S] = a.E;
  }
}

// band widths per packed state (for the band offset scan)
__global__ void __launch_bounds__(256) k_gp_band_counts2(GP a) {
  const int l = blockIdx.x;
  const int s0 = a.s_off[l], ns = a.s_off[l + 1] - s0;
  for (int n = blockIdx.y * blockDim.x + threadIdx.x; n < ns; n += gridDim.y * blockDim.x) {
    const int go = s0 + a.orig[s0 + n];
    const int hi = a.bhi[go];
    a.counts[s0 + n] = hi >= 0 ? hi - a.blo[go] + 1 : 0;
  }
}

// grid (L, tiles): +1 at the first frame of every word arc, -1 at the frame after its last one
// (two atomics per arc, not one per arc x frame); k_gp_frame_counts turns the differences into the
// arcs alive in every frame
__global__ void __launch_bounds__(256) k_gp_frames(GP a) {
  // (lattice-fastest grid on purpose: tile-fastest puts the CTAs in flight on the same few lattices'
  // frame counters and the atomics collide -- 5.8 vs 10.1 ms)
  const int l = blockIdx.x;
  const int e0 = a.e_off[l], e1 = a.e_off[l + 1];
  const int T = a.fr_base[l + 1] - a.fr_base[l] - 1;
  int32_t* cnt = a.fr_cnt + a.fr_base[l];
  // consecutive arcs leave the same state, i.e. start in the same frame (and mostly end in one of a
  // few): the lanes of a warp are grouped by frame and one atomic per group is issued
  const int lane = threadIdx.x & 31;
  for (int p0 = e0 + blockIdx.y * blockDim.x; p0 < e1; p0 += gridDim.y * blockDim.x) {
    const int p = p0 + threadIdx.x;
    int fa = -1, fb = -1;
    if (p < e1) {
      const int4 r = a.out_rec[p];
      if (r.w != 0) {
        const int x = max(a.ptime[a.out_src[p]], 0), y = min(a.ptime[r.x], T);
        if (y > x) {
          fa = x;
          fb = y;  // fb <= T: the slot that closes the lattice takes the last ones
        }
      }
    }
    const unsigned int ga = __match_any_sync(0xffffffffu, fa), gb = __match_any_sync(0xffffffffu, fb);
    if (fa >= 0 && lane == __ffs(ga) - 1) atomicAdd(cnt + fa, __popc(ga));
    if (fb >= 0 && lane == __ffs(gb) - 1) atomicAdd(cnt + fb, -__popc(gb));
  }
}

// one CTA per lattice: in-place inclusive scan of the frame slots (T + 1 of them)
__global__ void __launch_bounds__(256) k_gp_frame_counts(GP a) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = blockIdx.x;
  const int n = a.fr_base[l + 1] - a.fr_base[l];
  int32_t* cnt = a.fr_cnt + a.fr_base[l];
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = 0; tile < n; tile += 256) {
    const int i = tile + tid;
    const int v = i < n ? cnt[i] : 0;
    const int pre = cta_exclusive_scan<int, 256>(v, warp_sum, carry_s);
    if (i < n) cnt[i] = pre + v;
  }
}

int h2d(klu_ctx* c, void* dst, const void* src, size_t bytes) {
  if (bytes) KLU_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
  return 0;
}

int upload(klu_ctx* c, DevBuf& b, const void* src, size_t bytes) {
  KLU_TRY(b.reserve(bytes ? bytes : 16));
  return h2d(c, b.p, src, bytes);
}

}  // namespace

int pack_and_upload_gpu(klu_ctx* c, const klu_lattices* in) {
  const int32_t L = in->num_lattices;
  if (L < 0) {
    set_error("klu_load: negative lattice count");
    return 1;
  }
  if (L && (in->state_off[0] != 0 || in->arc_off[0] != 0)) {
    set_error("klu_load: offsets must start at 0");
    return 1;
  }
  const int64_t S = L ? in->state_off[L] : 0, E = L ? in->arc_off[L] : 0;
  if (S >= ((int64_t)1 << 31) - 2 || E >= ((int64_t)1 << 31) - 2) {
    set_error("klu_load: batch too large for 32-bit indices; split it");
    return 1;
  }
  const size_t S1 = (size_t)std::max<int64_t>(S, 1), E1 = (size_t)std::max<int64_t>(E, 1);
  // ---- raw input on the device (scratch slots are free while loading) ----
  std::vector<int32_t> s_off(L + 1), e_off(L + 1), order(L);
  for (int32_t l = 0; l <= L; ++l) {
    s_off[l] = (int32_t)in->state_off[l];
    e_off[l] = (int32_t)in->arc_off[l];
  }
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int32_t x, int32_t y) {
    return (in->arc_off[x + 1] - in->arc_off[x]) > (in->arc_off[y + 1] - in->arc_off[y]);
  });
  DevBuf* sc = c->d_scratch;
  enum { R_SRC = 0, R_DST, R_LABEL, R_DUR, R_G, R_A, R_KEYA, R_KEYB, R_VALA, R_VALB, R_MISC, R_MISC2 };
  // Host-to-device copies of different contexts take turns (one process-wide lock held
  // until this batch's copies have landed): with several contexts on one GPU -- the
  // tools' worker threads, a pipelined caller -- the next batch's upload then overlaps
  // this batch's packing, run and result download instead of interleaving with its upload.
  static std::mutex h2d_turn;
  KLU_TRY(stage_begin(c, (size_t)L));
  klu_trace(c, "load: waiting for the upload turn");
  std::unique_lock<std::mutex> h2d_lock(h2d_turn);
  klu_trace(c, "load: upload begins");
  timespec up0;
  clock_gettime(CLOCK_MONOTONIC, &up0);
  KLU_TRY(upload(c, c->d_s_off, s_off.data(), 4 * (size_t)(L + 1)));
  KLU_TRY(upload(c, c->d_e_off, e_off.data(), 4 * (size_t)(L + 1)));
  KLU_TRY(upload(c, c->d_order, order.data(), 4 * (size_t)L));
  if (in->arc_src) KLU_TRY(upload(c, sc[R_SRC], in->arc_src, 4 * (size_t)E));
  else KLU_TRY(sc[R_SRC].reserve(4 * E1));
  if (in->arc_dst) KLU_TRY(upload(c, sc[R_DST], in->arc_dst, 4 * (size_t)E));
  else {
    KLU_TRY(sc[R_DST].reserve(4 * E1));
    KLU_TRY(upload(c, sc[R_KEYB], in->arc_dst_delta_u16, 2 * (size_t)E));  // expanded on the device below
  }
  if (in->arc_label) KLU_TRY(upload(c, sc[R_LABEL], in->arc_label, 4 * (size_t)E));
  else {
    KLU_TRY(sc[R_LABEL].reserve(4 * E1));
    KLU_TRY(upload(c, sc[R_VALA], in->arc_label_u16, 2 * (size_t)E));
  }
  if (in->arc_dur) KLU_TRY(upload(c, sc[R_DUR], in->arc_dur, 4 * (size_t)E));
  else {
    KLU_TRY(sc[R_DUR].reserve(4 * E1));
    KLU_TRY(upload(c, sc[R_KEYA], in->arc_dur_u8, (size_t)E));
  }
  KLU_TRY(upload(c, sc[R_G], in->arc_graph, 4 * (size_t)E));
  KLU_TRY(upload(c, sc[R_A], in->arc_acoustic, 4 * (size_t)E));
  // per-state raw input + per-state work arrays share one allocation:
  // fg, fa, fdur, first_arc(+1), level, time, blo, bhi, counts  (9 x S + 1 ints)
  KLU_TRY(sc[R_MISC].reserve(4 * (10 * S1 + 16)));
  int32_t* misc = sc[R_MISC].as<int32_t>();
  float* r_fg = reinterpret_cast<float*>(misc);
  float* r_fa = reinterpret_cast<float*>(misc + S1);
  int32_t* r_fdur = misc + 2 * S1;
  if (S) {
    KLU_TRY(h2d(c, r_fg, in->fin_graph, 4 * (size_t)S));
    KLU_TRY(h2d(c, r_fa, in->fin_acoustic, 4 * (size_t)S));
    if (in->fin_dur) KLU_TRY(h2d(c, r_fdur, in->fin_dur, 4 * (size_t)S));
  }
  // (per-state arc counts, when the caller gave those instead of arc sources: counts slot of misc)
  if (!in->arc_src) KLU_TRY(h2d(c, misc + 8 * S1 + 8, in->state_num_arcs, 4 * (size_t)S));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  {
    timespec up1;
    clock_gettime(CLOCK_MONOTONIC, &up1);
    c->load_upload_ms = (float)((up1.tv_sec - up0.tv_sec) * 1e3 + (up1.tv_nsec - up0.tv_nsec) * 1e-6);
  }
  h2d_lock.unlock();
  klu_trace(c, "load: upload done, packing");
  KLU_CUDA(cudaEventRecord(c->ev_p0, c->stream));
  // per-lattice metadata: meta (L x 8 int), cap (2L int64), lat_tot (L+1 int64), where flags
  KLU_TRY(sc[R_MISC2].reserve(4 * (size_t)M_STRIDE * (L + 1) + 8 * (size_t)(3 * L + 4) + 2 * (size_t)L + 64));
  char* m2 = sc[R_MISC2].as<char>();
  KLU_CUDA(cudaMemsetAsync(m2, 0, sc[R_MISC2].cap, c->stream));
  KLU_TRY(c->d_counter.reserve(64));
  KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));

  GP a;
  memset(&a, 0, sizeof(a));
  a.L = L;
  a.S = (int)S;
  a.E = (int)E;
  a.s_off = c->d_s_off.as<int32_t>();
  a.e_off = c->d_e_off.as<int32_t>();
  a.src = sc[R_SRC].as<int32_t>();
  a.dst = sc[R_DST].as<int32_t>();
  a.label = sc[R_LABEL].as<int32_t>();
  a.dur = sc[R_DUR].as<int32_t>();
  a.g = sc[R_G].as<float>();
  a.a = sc[R_A].as<float>();
  a.fg = r_fg;
  a.fa = r_fa;
  a.fdur = in->fin_dur ? r_fdur : nullptr;
  a.first_arc = misc + 3 * S1;  // S + 1 entries
  a.level = misc + 4 * S1 + 8;
  a.time = misc + 5 * S1 + 8;
  a.blo = misc + 6 * S1 + 8;
  a.bhi = misc + 7 * S1 + 8;
  a.counts = misc + 8 * S1 + 8;
  a.meta = reinterpret_cast<int32_t*>(m2);
  a.cap = reinterpret_cast<long long*>(m2 + 4 * (size_t)M_STRIDE * (L + 1));
  a.lat_tot = a.cap + 2 * (size_t)L + 2;
  unsigned char* where = reinterpret_cast<unsigned char*>(a.lat_tot + L + 2);

  c->L = L;
  c->S = S;
  c->E = E;
  c->h_s_off.assign(in->state_off, in->state_off + L + 1);
  c->h_e_off.assign(in->arc_off, in->arc_off + L + 1);
  c->h_num_frames.assign(L, 0);
  c->h_maxtime.assign(L, 0);
  c->h_times_ok.assign(L, 1);
  c->h_cap_frame.assign(L, 0);
  c->h_cap_pos.assign(L, 0);
  c->h_maxlen.assign(L, 0);
  c->h_band_off.assign(L + 1, 0);
  c->h_fr_base.assign(L + 1, 0);
  c->h_new2old.clear();
  c->h_old2new.clear();
  c->max_label = c->max_time = c->max_len = c->max_indeg = c->max_outdeg = c->max_states = c->max_span = 0;
  c->avg_deg = S ? (double)E / (double)S : 0.0;
  c->band_total = 0;
  c->frame_entries = 0;
  c->NL = 0;
  // packed per-state / per-arc outputs
  KLU_TRY(c->d_in_rec.reserve(16 * E1));
  KLU_TRY(c->d_out_rec.reserve(16 * E1));
  KLU_TRY(c->d_in_off.reserve(4 * (S1 + 1)));
  KLU_TRY(c->d_out_off.reserve(4 * (S1 + 1)));
  KLU_TRY(c->d_out_src.reserve(4 * E1));
  KLU_TRY(c->d_out_orig.reserve(4 * E1));
  KLU_TRY(c->d_in2out.reserve(4 * E1));
  KLU_TRY(c->d_fin_g.reserve(4 * S1));
  KLU_TRY(c->d_fin_a.reserve(4 * S1));
  KLU_TRY(c->d_time.reserve(4 * S1));
  KLU_TRY(c->d_orig.reserve(4 * S1));
  KLU_TRY(c->d_level.reserve(4 * S1));
  KLU_TRY(c->d_band_lo.reserve(4 * S1));
  KLU_TRY(c->d_band_off.reserve(8 * (S1 + 1)));
  KLU_TRY(c->d_old2new.reserve(4 * S1));
  KLU_TRY(c->d_lvl_off.reserve(4 * (size_t)(L + 1)));
  KLU_TRY(c->d_lvl_start.reserve(4 * (S1 + (size_t)L + 1)));
  KLU_TRY(c->d_fr_base.reserve(4 * (size_t)(L + 1)));
  if (L == 0) {
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  }
  int64_t max_arcs = 0, max_states = 0;
  for (int32_t l = 0; l < L; ++l) {
    max_arcs = std::max(max_arcs, in->arc_off[l + 1] - in->arc_off[l]);
    max_states = std::max(max_states, in->state_off[l + 1] - in->state_off[l]);
  }
  c->max_states = (int32_t)max_states;
  const int arc_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  const int st_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_states + 255) / 256, 16));
  if (!in->arc_src) {  // arcs grouped by source state: expand the sources from the per-state arc counts
    {
      KLU_LAUNCH(c, "k_gp_lat_scan");
      k_gp_lat_scan<0><<<L, 256, 0, c->stream>>>(a.counts, a.s_off, a.e_off, a.first_arc, nullptr, nullptr);
    }
    KLU_TRY(check_launch("k_gp_lat_scan(src)"));
    {
      KLU_LAUNCH(c, "k_gp_expand_src");
      k_gp_expand_src<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a, sc[R_SRC].as<int32_t>());
    }
    KLU_TRY(check_launch("k_gp_expand_src"));
  }
  if (!in->arc_dst || !in->arc_dur || !in->arc_label) {
    KLU_LAUNCH(c, "k_gp_expand_compact");
    k_gp_expand_compact<<<c->num_sms * 8, 256, 0, c->stream>>>(
        in->arc_dur ? nullptr : sc[R_KEYA].as<uint8_t>(), in->arc_dst ? nullptr : sc[R_KEYB].as<uint16_t>(),
        in->arc_label ? nullptr : sc[R_VALA].as<uint16_t>(), sc[R_SRC].as<int32_t>(), sc[R_DUR].as<int32_t>(),
        sc[R_DST].as<int32_t>(), sc[R_LABEL].as<int32_t>(), E);
    KLU_TRY(check_launch("k_gp_expand_compact"));
  }
  {
    KLU_LAUNCH(c, "k_gp_first_arc");
    k_gp_first_arc<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_gp_first_arc"));
  {
    KLU_LAUNCH(c, "k_gp_levels");
    // (a variant with the per-state work arrays in shared memory, one warp per CTA, measured no
    // faster: 49 against 46 ms of packing per 10 k c2 lattices -- the walk is bound by its ns
    // dependent steps, not by where the arrays live)
    const int grid = std::max(1, std::min((L + 3) / 4, c->num_sms * 16));
    k_gp_levels<<<grid, 128, 0, c->stream>>>(a, c->d_counter.as<int>());
  }
  KLU_TRY(check_launch("k_gp_levels"));
  // ---- host round trip 1: per-lattice metadata ----
  std::vector<int32_t> meta((size_t)M_STRIDE * L);
  KLU_TRY(small_d2h(c, meta.data(), a.meta, 4 * meta.size()));
  KLU_TRY(small_sync(c));
  klu_trace(c, "load: levels known");
  std::vector<int32_t> lvl_off(L + 1, 0);
  for (int32_t l = 0; l < L; ++l) {
    const int32_t* m = meta.data() + (size_t)M_STRIDE * l;
    if (m[M_ERR] == 1) {
      set_error("klu_load: lattice " + std::to_string(l) +
                ": arcs must be grouped by ascending src and topologically sorted (src < dst)");
      return 1;
    }
    if (m[M_ERR] == 2) {
      set_error("klu_load: lattice " + std::to_string(l) + ": non-finite arc weight");
      return 1;
    }
    lvl_off[l + 1] = lvl_off[l] + m[M_NL] + 1;
    c->h_fr_base[l + 1] = c->h_fr_base[l] + m[M_FRAMES] + 1;
    c->h_num_frames[l] = m[M_FRAMES];
    c->h_maxtime[l] = m[M_MAXTIME];
    c->h_times_ok[l] = (uint8_t)m[M_TIMES_OK];
    c->h_maxlen[l] = m[M_MAXLEN];
    c->max_label = std::max(c->max_label, m[M_MAXLABEL]);
    c->max_time = std::max(c->max_time, m[M_MAXTIME]);
    c->max_len = std::max(c->max_len, m[M_MAXLEN]);
  }
  c->NL = lvl_off[L] - L;
  KLU_TRY(upload(c, c->d_lvl_off, lvl_off.data(), 4 * (size_t)(L + 1)));
  KLU_TRY(upload(c, c->d_fr_base, c->h_fr_base.data(), 4 * (size_t)(L + 1)));
  const size_t F1 = (size_t)c->h_fr_base[L] + 2;
  KLU_TRY(c->d_fr_off.reserve(8 * F1));
  a.old2new = c->d_old2new.as<int32_t>();
  a.orig = c->d_orig.as<int32_t>();
  a.plevel = c->d_level.as<int32_t>();
  a.ptime = c->d_time.as<int32_t>();
  a.band_lo = c->d_band_lo.as<int32_t>();
  a.lvl_start = c->d_lvl_start.as<int32_t>();
  a.in_off = c->d_in_off.as<int32_t>();
  a.out_off = c->d_out_off.as<int32_t>();
  a.out_src = c->d_out_src.as<int32_t>();
  a.out_orig = c->d_out_orig.as<int32_t>();
  a.in2out = c->d_in2out.as<int32_t>();
  a.lvl_off = c->d_lvl_off.as<int32_t>();
  a.fr_base = c->d_fr_base.as<int32_t>();
  a.pfg = c->d_fin_g.as<float>();
  a.pfa = c->d_fin_a.as<float>();
  a.band_off = c->d_band_off.as<int64_t>();
  a.fr_off = c->d_fr_off.as<int64_t>();
  a.in_rec = c->d_in_rec.as<int4>();
  a.out_rec = c->d_out_rec.as<int4>();
  // ---- states: stable sort by level ----
  const size_t NK = std::max(S1, E1);
  KLU_TRY(sc[R_KEYA].reserve(8 * NK));
  KLU_TRY(sc[R_KEYB].reserve(8 * NK));
  KLU_TRY(sc[R_VALA].reserve(4 * NK));
  KLU_TRY(sc[R_VALB].reserve(4 * NK));
  // 64-bit segment bases for the sort
  KLU_TRY(c->d_res[6].reserve(8 * (size_t)(2 * L + 2)));
  int64_t* seg64 = c->d_res[6].as<int64_t>();
  KLU_TRY(small_h2d(c, seg64, in->state_off, 8 * (size_t)(L + 1)));
  KLU_TRY(small_h2d(c, seg64 + L + 1, in->arc_off, 8 * (size_t)(L + 1)));
  KLU_TRY(c->d_res[7].reserve(4 * (size_t)(2 * L + 2)));
  std::vector<int32_t> seg_cnt(2 * (size_t)L);
  for (int32_t l = 0; l < L; ++l) {
    seg_cnt[l] = (int32_t)(in->state_off[l + 1] - in->state_off[l]);
    seg_cnt[L + l] = (int32_t)(in->arc_off[l + 1] - in->arc_off[l]);
  }
  KLU_TRY(small_h2d(c, c->d_res[7].p, seg_cnt.data(), 4 * seg_cnt.size()));
  unsigned long long* key_a = sc[R_KEYA].as<unsigned long long>();
  unsigned long long* key_b = sc[R_KEYB].as<unsigned long long>();
  unsigned int* val_a = sc[R_VALA].as<unsigned int>();
  unsigned int* val_b = sc[R_VALB].as<unsigned int>();
  {
    KLU_LAUNCH(c, "k_gp_state_keys");
    k_gp_state_keys<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a, key_a, val_a);
  }
  KLU_TRY(check_launch("k_gp_state_keys"));
  SegSortArgs ss;
  ss.seg_base = seg64;
  ss.seg_cnt = c->d_res[7].as<int32_t>();
  ss.key_a = key_a;
  ss.val_a = val_a;
  ss.key_b = key_b;
  ss.val_b = val_b;
  ss.where = where;
  ss.lo_bit = 0;
  ss.hi_bit = 32;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, ss, L, (int64_t)S));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(states)"));
  {
    KLU_LAUNCH(c, "k_gp_state_perm");
    k_gp_state_perm<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a, key_a, key_b, val_a, val_b, where);
  }
  KLU_TRY(check_launch("k_gp_state_perm"));
  // out_off = e_off[l] + scan(out-degree in packed order)
  {
    KLU_LAUNCH(c, "k_gp_lat_scan");
    k_gp_lat_scan<0><<<L, 256, 0, c->stream>>>(a.counts, a.s_off, a.e_off, a.out_off, nullptr, nullptr);
  }
  KLU_TRY(check_launch("k_gp_lat_scan(out)"));
  // ---- arcs: source order by block move, destination order by stable sort ----
  {
    KLU_LAUNCH(c, "k_gp_scatter");
    k_gp_scatter<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a, reinterpret_cast<unsigned int*>(key_a), val_a);
  }
  KLU_TRY(check_launch("k_gp_scatter"));
  SegSortArgs32 sa;  // keys = lattice-local destination states: as many bits as the largest lattice needs
  sa.seg_base = seg64 + L + 1;
  sa.seg_cnt = c->d_res[7].as<int32_t>() + L;
  sa.key_a = reinterpret_cast<unsigned int*>(key_a);
  sa.key_b = reinterpret_cast<unsigned int*>(key_b);
  sa.val_a = val_a;
  sa.val_b = val_b;
  sa.where = where;
  sa.lo_bit = 0;
  {
    int64_t max_ns = 1;
    for (int32_t l = 0; l < L; ++l) max_ns = std::max<int64_t>(max_ns, in->state_off[l + 1] - in->state_off[l]);
    sa.hi_bit = 1;
    while (sa.hi_bit < 32 && ((int64_t)1 << sa.hi_bit) < max_ns) ++sa.hi_bit;
  }
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, sa, L, (int64_t)E));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(arcs)"));
  {
    KLU_LAUNCH(c, "k_gp_in_build");
    k_gp_in_build<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a, sa.key_a, sa.key_b, val_a, val_b, where);
  }
  KLU_TRY(check_launch("k_gp_in_build"));
  // ---- band offsets: per-lattice scan + lattice bases ----
  {
    KLU_LAUNCH(c, "k_gp_band_counts");
    k_gp_band_counts2<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_gp_band_counts"));
  {
    KLU_LAUNCH(c, "k_gp_lat_scan");
    k_gp_lat_scan<1><<<L, 256, 0, c->stream>>>(a.counts, a.s_off, nullptr, nullptr, a.band_off, a.lat_tot);
  }
  KLU_TRY(check_launch("k_gp_lat_scan(band)"));
  KLU_TRY(scan_counts(c, a.lat_tot, 0, L, a.lat_tot, "k_gp_scan_tot"));
  {
    KLU_LAUNCH(c, "k_gp_add_base");
    k_gp_add_base<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a.band_off, a.s_off, a.lat_tot, L, a.band_off + S);
  }
  KLU_TRY(check_launch("k_gp_add_base(band)"));
  // ---- host round trip 2: band bases and expansion capacities ----
  std::vector<long long> h_tot(L + 1), h_cap(2 * (size_t)L);
  KLU_TRY(small_d2h(c, h_tot.data(), a.lat_tot, 8 * (size_t)(L + 1)));
  KLU_TRY(small_d2h(c, h_cap.data(), a.cap, 16 * (size_t)L));
  KLU_TRY(small_d2h(c, &c->max_span, a.meta + (size_t)L * M_STRIDE, 4));
  KLU_TRY(small_sync(c));
  klu_trace(c, "load: bands known");
  for (int32_t l = 0; l <= L; ++l) c->h_band_off[l] = h_tot[l];
  c->band_total = h_tot[L];
  std::vector<long long> fa_base(L + 1, 0);
  for (int32_t l = 0; l < L; ++l) {
    c->h_cap_frame[l] = h_cap[2 * l];
    c->h_cap_pos[l] = h_cap[2 * l + 1];
    fa_base[l + 1] = fa_base[l] + h_cap[2 * l];
  }
  c->frame_entries = fa_base[L];
  c->frame_ready = false;  // the frame index (lattice-to-word-frame-post only) is built on first use
  KLU_CUDA(cudaEventRecord(c->ev_p1, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // host-side vectors used by async copies die here
  cudaEventElapsedTime(&c->load_pack_ms, c->ev_p0, c->ev_p1);
  klu_trace(c, "load: packed");
  return 0;
}

// The frame index of lattice-to-word-frame-post (frame -> arc CSR offsets, then the (frame, word)
// groups of klu_frame.cu): built from the packed batch the first time a frame-post run asks
// for it, so the other tools' loads do not pay for it.  Its device time is reported with the
// load's (klu_load_times).
int ensure_frame_index(klu_ctx* c) {
  if (c->frame_ready) return 0;
  const int32_t L = c->L;
  c->lazy_pack_ms = 0.f;
  if (L == 0) {
    c->frame_ready = true;
    return build_frame_groups(c);
  }
  KLU_CUDA(cudaEventRecord(c->ev_p0, c->stream));
  DevBuf* sc = c->d_scratch;
  enum { R_VALB = 9, R_MISC2 = 11 };
  GP a;
  memset(&a, 0, sizeof(a));
  a.L = L;
  a.S = (int)c->S;
  a.E = (int)c->E;
  a.s_off = c->d_s_off.as<int32_t>();
  a.e_off = c->d_e_off.as<int32_t>();
  a.fr_base = c->d_fr_base.as<int32_t>();
  a.out_rec = c->d_out_rec.as<int4>();
  a.out_src = c->d_out_src.as<int32_t>();
  a.ptime = c->d_time.as<int32_t>();
  const size_t F1 = (size_t)c->h_fr_base[L] + 2;
  KLU_TRY(c->d_fr_off.reserve(8 * F1));
  a.fr_off = c->d_fr_off.as<int64_t>();
  KLU_TRY(sc[R_MISC2].reserve(8 * (size_t)(2 * L + 4)));
  a.lat_tot = sc[R_MISC2].as<long long>();
  a.cap = a.lat_tot + L + 2;
  std::vector<long long> fa_base(L + 1, 0);
  int64_t max_arcs = 0, max_frames = 0;
  for (int32_t l = 0; l < L; ++l) {
    fa_base[l + 1] = fa_base[l] + c->h_cap_frame[l];
    max_arcs = std::max(max_arcs, c->h_e_off[l + 1] - c->h_e_off[l]);
    max_frames = std::max<int64_t>(max_frames, c->h_fr_base[l + 1] - c->h_fr_base[l]);
  }
  const int arc_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  const int st_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_frames + 255) / 256, 16));
  KLU_TRY(stage_begin(c, (size_t)L));
  // ---- frame -> arc CSR ----
  KLU_TRY(c->d_frame_arc.reserve(4 * (size_t)std::max<long long>(fa_base[L], 1)));
  a.frame_arc = c->d_frame_arc.as<int32_t>();
  KLU_TRY(sc[R_VALB].reserve(4 * F1));  // frame counters (the sort buffers are free again)
  a.fr_cnt = sc[R_VALB].as<int32_t>();
  KLU_CUDA(cudaMemsetAsync(a.fr_cnt, 0, 4 * F1, c->stream));
  KLU_TRY(small_h2d(c, a.lat_tot, fa_base.data(), 8 * (size_t)(L + 1)));
  {
    KLU_LAUNCH(c, "k_gp_frames");
    k_gp_frames<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_gp_frames(count)"));
  {
    KLU_LAUNCH(c, "k_gp_frame_counts");
    k_gp_frame_counts<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_gp_frame_counts"));
  {
    // frame slots of lattice l: fr_base[l] .. fr_base[l+1]-1 (the last one closes the lattice)
    KLU_LAUNCH(c, "k_gp_lat_scan");
    k_gp_lat_scan<1><<<L, 256, 0, c->stream>>>(a.fr_cnt, a.fr_base, nullptr, nullptr, a.fr_off, a.cap /*unused totals*/);
  }
  KLU_TRY(check_launch("k_gp_lat_scan(frames)"));
  {
    KLU_LAUNCH(c, "k_gp_add_base");
    k_gp_add_base<<<dim3(L, st_tiles), 256, 0, c->stream>>>(a.fr_off, a.fr_base, a.lat_tot, L,
                                                            a.fr_off + c->h_fr_base[L]);
  }
  KLU_TRY(check_launch("k_gp_add_base(frames)"));
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // fa_base is read by a staged copy
  klu_trace(c, "frame index: offsets built, building the (frame, word) groups");
  KLU_TRY(build_frame_groups(c));
  KLU_CUDA(cudaEventRecord(c->ev_p1, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->lazy_pack_ms, c->ev_p0, c->ev_p1);
  c->frame_ready = true;
  return 0;
}

}  // namespace klu
