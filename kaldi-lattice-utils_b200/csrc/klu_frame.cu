// klu_frame.cu -- frame-synchronous word posteriorgram (SURVEY.md F1, K6-K8 fused).
//
// Reference: latbin/lattice-to-word-frame-post.cc:94-135 -- for every word arc and
// every frame k it spans, acc[k][word] (a std::map per frame) is LogAdd-ed with
// fw[u] + bw[v] - (float)(g + a); then each frame is normalised, cast to float and
// sorted by (float log-posterior desc, word asc).
//
// Which (frame, word) groups exist, which arcs feed each of them and how many rows
// every frame emits depends only on labels and state times, not on the weights.
// So klu_load() builds that structure ONCE per batch (build_frame_groups): the arcs
// numbered by start time, the arc x frame instances of a lattice sorted by (frame,
// word, arc), a head bit on the first instance of every group, and the dense output
// offset of every frame.  A run is then the log sweeps and two kernels:
//   k_frame_groups  one CTA per run of kFramesPerItem frames: the posterior
//                   exp(fw[u] + bw[v] - cost - total) of every arc of the run's
//                   window into shared memory (f64; exp(-700) ~ 1e-304 is the
//                   underflow horizon), then one THREAD per (frame, word) group adds
//                   the posteriors of the group's instances in arc order and writes
//                   (float)log(sum) to the group's pre-order row;
//   k_frame_order   one warp per run of frames: orders the frame's rows in shared
//                   memory (bitonic, key = ~ordered float bits << 32 | word) and
//                   writes (word, logp) to the dense table in place.
// A group whose sum underflows (or is empty) is redone exactly in the log domain
// from alpha/beta (exact_group_logp); frames with more groups than the shared-memory
// order buffer holds are ordered in global memory (slow, same results).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

constexpr int kFrameWarps = 4;      // warps per CTA
constexpr int kGroupCap = 256;      // rows of one frame ordered in shared memory
constexpr int kFramesPerItem = 16;  // consecutive frames handled by one warp
constexpr int kDeferMin = 4;        // groups longer than this are summed in a second pass
constexpr int kLongCap = 1024;      // ... at most this many per run of frames (the rest are summed in place)

struct FrameArgs {
  BatchView b;
  CostParams cp;
  const double* alpha;
  const double* beta;
  const double* total;
  const int32_t* item_base;  // [L+1] first work item of each lattice
  int num_items;
  const int64_t* gloc;       // per frame slot: lattice-local first output row (T+1 per lattice)
  const int64_t* res_off;    // [L+1] first output row of each lattice
  const int32_t* gwords;     // word of every (frame, word) group, in pre-order row order (static)
  const uint32_t* gstart;    // [rows + 1] first instance of every group (static)
  const int4* tarc;          // [E] arcs in START-TIME order: {src, dst, graph bits, acoustic bits} (static)
  const int32_t* tlabel;     // [E] their labels; frame_arc holds indices into this order
  const int32_t* run_lo;     // per work item (run of frames): smallest / largest time-order arc index among
  const int32_t* run_hi;     // its instances (static); the arcs in between are the run's "window"
  int win_cap;               // window entries that fit the dynamic shared memory
  int32_t* o_word;
  float* o_logp;
};

__device__ __forceinline__ float inv_ord_f32(unsigned int u) {
  const unsigned int b = (u & 0x80000000u) ? (u ^ 0x80000000u) : ~u;
  return __uint_as_float(b);
}

// fw[u] + bw[next] - (float)(g + a), latbin/lattice-to-word-frame-post.cc:102-104
__device__ __forceinline__ double arc_value(const FrameArgs& a, int j) {  // j: time-order arc index
  const int4 t = __ldg(a.tarc + j);
  const int4 r = make_int4(t.y, t.z, t.w, __ldg(a.tlabel + j));
  return __dadd_rn(__dadd_rn(a.alpha[t.x], a.beta[t.y]), -rec_cost(r, a.cp));
}

// Exact log-posterior of the group that ENDS at instance `iend` of a frame's list
// (walks back to the group's head): max first, then libm exp / log.
__device__ __noinline__ double exact_group_logp(const FrameArgs& a, const int32_t* fa, int iend, double total) {
  double m = neg_inf();
  for (int q = iend;; --q) {
    const unsigned int w = (unsigned int)fa[q];
    m = fmax(m, arc_value(a, (int)(w & 0x7fffffffu)));
    if (w >> 31) break;
  }
  if (!(m > neg_inf())) return neg_inf();
  if (m == pos_inf()) return pos_inf();
  double s = 0.0;
  for (int q = iend;; --q) {
    const unsigned int w = (unsigned int)fa[q];
    s += exp(arc_value(a, (int)(w & 0x7fffffffu)) - m);
    if (w >> 31) break;
  }
  return (m + log(s)) - total;
}

// Warp-wide bitonic sort of N keys in shared memory (ascending), N a compile-time
// power of two: every stage is unrolled, so the pair indices are a couple of bit
// operations on the lane id.  For N >= 128 a lane handles TWO adjacent compare-
// exchange pairs per step through 16-byte shared-memory accesses.
template <int N>
__device__ __forceinline__ void warp_bitonic_fixed(unsigned long long* keys, int lane) {
#pragma unroll
  for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (N >= 128 && j >= 2) {
#pragma unroll
        for (int t = 0; t < N / 128; ++t) {
          const int p0 = (lane + 32 * t) << 1;  // even pair index: pairs p0 and p0 + 1 sit side by side
          const int i = ((p0 & ~(j - 1)) << 1) | (p0 & (j - 1));
          const int q = i | j;
          const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(keys + i);
          const ulonglong2 y = *reinterpret_cast<const ulonglong2*>(keys + q);
          const bool up = (i & k) == 0;
          if ((x.x > y.x) == up) {
            keys[i] = y.x;
            keys[q] = x.x;
          }
          if ((x.y > y.y) == up) {
            keys[i + 1] = y.y;
            keys[q + 1] = x.y;
          }
        }
      } else if (N >= 128) {  // j == 1: the pair is one aligned 16-byte word
#pragma unroll
        for (int t = 0; t < N / 64; ++t) {
          const int i = (lane + 32 * t) << 1;
          const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(keys + i);
          const bool up = (i & k) == 0;
          if ((x.x > x.y) == up) *reinterpret_cast<ulonglong2*>(keys + i) = make_ulonglong2(x.y, x.x);
        }
      } else {
        if (lane < N / 2) {
          const int i = ((lane & ~(j - 1)) << 1) | (lane & (j - 1));
          const int q = i | j;
          const unsigned long long x = keys[i], y = keys[q];
          const bool up = (i & k) == 0;
          if ((x > y) == up) {
            keys[i] = y;
            keys[q] = x;
          }
        }
      }
      __syncwarp();
    }
  }
}


// slow path: odd-even transposition sort of a frame's (logp, word) rows in global memory
__device__ void warp_sort_rows_global(float* logp, int32_t* word, int n, int lane) {
  for (int round = 0; round < n; ++round) {
    for (int i = (round & 1) + 2 * lane; i + 1 < n; i += 64) {
      const unsigned long long x = ((unsigned long long)(~ord_f32(logp[i])) << 32) | (unsigned int)word[i];
      const unsigned long long y = ((unsigned long long)(~ord_f32(logp[i + 1])) << 32) | (unsigned int)word[i + 1];
      if (x > y) {
        const float tl = logp[i];
        logp[i] = logp[i + 1];
        logp[i + 1] = tl;
        const int32_t tw = word[i];
        word[i] = word[i + 1];
        word[i + 1] = tw;
      }
    }
    __syncwarp();
  }
}


// Fused arc posteriors + group sums for one run of kFramesPerItem frames per CTA.
// With the arcs numbered by start time (a copy made at pack time), the word arcs alive
// in a run of frames are a contiguous index range -- the run's window.  Phase 1 computes the posterior of
// every arc of the window into shared memory (coalesced record reads, one exp per arc;
// windows of neighbouring runs overlap by the arcs that span the boundary, ~1/8 extra);
// phase 2 adds each (frame, word) group's posteriors, one thread per group, from shared
// memory.  No per-arc posterior array in HBM, no dependent global gathers.  Runs whose window does not fit
// (very long arcs) take the posteriors from alpha/beta directly, instance by instance.
__global__ void __launch_bounds__(128) k_frame_groups(const __grid_constant__ FrameArgs a) {
  extern __shared__ double s_post[];
  const BatchView& b = a.b;
  const int item = blockIdx.x;
  const int l = last_le(a.item_base, 0, b.L - 1, item);  // lattice of this item
  const int T = b.fr_base[l + 1] - b.fr_base[l] - 1;
  const int k0 = (item - a.item_base[l]) * kFramesPerItem;
  const int k1 = min(T, k0 + kFramesPerItem);
  const int64_t* gl = a.gloc + b.fr_base[l];
  const int64_t row0 = a.res_off[l] + gl[k0], row1 = a.res_off[l] + gl[k1];
  if (row0 == row1) return;
  const int wlo = a.run_lo[item], whi = a.run_hi[item];
  const bool windowed = whi - wlo < a.win_cap;
  const double total = a.total[l];
  __shared__ int s_long[kLongCap];
  __shared__ int s_nlong;
  if (threadIdx.x == 0) s_nlong = 0;  // ordered before its first use by the barrier after phase 1
  if (windowed && threadIdx.x >= 96) {
    // the last warp first asks L2 for what phase 2 will read -- the run's group offsets
    // and instance ids, two contiguous ranges -- so that those loads, which sit on a
    // dependent chain (offset -> id -> shared-memory posterior), find them there
    const int pl = threadIdx.x - 96;
    const char* q = reinterpret_cast<const char*>(a.gstart + row0);
    const int64_t qb = (row1 - row0 + 1) * 4;
    for (int64_t off = pl * 128; off < qb; off += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(q + off));
    const uint32_t ilo = __ldg(a.gstart + row0), ihi = __ldg(a.gstart + row1);
    q = reinterpret_cast<const char*>(b.frame_arc + ilo);
    const int64_t ib = (int64_t)(ihi - ilo) * 4;
    for (int64_t off = pl * 128; off < ib; off += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(q + off));
  }
  if (windowed) {
    // four arcs per thread and trip: their record, label and score loads go out together
    for (int j0 = wlo + threadIdx.x; j0 <= whi; j0 += 4 * blockDim.x) {
      int4 t[4];
      int lab[4];
      double al[4], be[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * blockDim.x;
        if (j <= whi) {
          t[u] = __ldg(a.tarc + j);
          lab[u] = __ldg(a.tlabel + j);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * blockDim.x;
        if (j <= whi) {
          al[u] = a.alpha[t[u].x];
          be[u] = a.beta[t[u].y];
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * blockDim.x;
        if (j <= whi) {
          const int4 r = make_int4(t[u].y, t[u].z, t[u].w, lab[u]);
          s_post[j - wlo] = lab[u] != 0 ? fast_exp(__dadd_rn(__dadd_rn(al[u], be[u]), -rec_cost(r, a.cp)) - total) : 0.0;
        }
      }
    }
    __syncthreads();
  }
  // two groups per thread and trip: both offset pairs, then both first id quads, are in flight together.
  // Groups of more than four instances (one in ten) would hold the other 31 lanes of
  // their warp in a long loop: they are put on a list in shared memory instead and
  // summed afterwards, long ones side by side.  A group is always added up by one
  // thread in instance order, so which thread does it cannot change the result.
  // (trip count uniform across a warp: the list push below is a warp-wide ballot)
  for (int64_t g0 = row0 + threadIdx.x; g0 - (threadIdx.x & 31) < row1; g0 += 2 * blockDim.x) {
    uint32_t i0[2], i1[2];
    double sum[2] = {0.0, 0.0};
    bool defer[2] = {false, false};
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int64_t g = g0 + v * blockDim.x;
      i0[v] = g < row1 ? __ldg(a.gstart + g) : 0u;
      i1[v] = g < row1 ? __ldg(a.gstart + g + 1) : 0u;
    }
    if (windowed) {
      int e[2][4];
#pragma unroll
      for (int v = 0; v < 2; ++v)
#pragma unroll
        for (int u = 0; u < 4; ++u)
          e[v][u] = i0[v] + u < i1[v] ? (int)((unsigned int)__ldg(b.frame_arc + i0[v] + u) & 0x7fffffffu) - wlo : -1;
#pragma unroll
      for (int v = 0; v < 2; ++v) {
#pragma unroll
        for (int u = 0; u < 4; ++u) sum[v] += e[v][u] >= 0 ? s_post[e[v][u]] : 0.0;
        const bool is_long = i1[v] - i0[v] > (unsigned int)kDeferMin;
        const unsigned int m = __ballot_sync(0xffffffffu, is_long);
        if (m) {
          const int lane = threadIdx.x & 31;
          int base = 0;
          if (lane == 0) base = atomicAdd(&s_nlong, __popc(m));
          base = __shfl_sync(0xffffffffu, base, 0);
          const int slot = base + __popc(m & ((1u << lane) - 1u));
          if (is_long && slot < kLongCap) {
            s_long[slot] = (int)(g0 + v * blockDim.x - row0);
            defer[v] = true;
          }
        }
        if (!defer[v])
          for (uint32_t i = i0[v] + 4; i < i1[v]; ++i)
            sum[v] += s_post[(int)((unsigned int)__ldg(b.frame_arc + i) & 0x7fffffffu) - wlo];
      }
    } else {
#pragma unroll
      for (int v = 0; v < 2; ++v)
        for (uint32_t i = i0[v]; i < i1[v]; ++i)
          sum[v] += fast_exp(arc_value(a, (int)((unsigned int)__ldg(b.frame_arc + i) & 0x7fffffffu)) - total);
    }
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int64_t g = g0 + v * blockDim.x;
      if (g < row1 && !defer[v]) {
        const double lp = sum[v] >= 1e-280 ? fast_log(sum[v]) : exact_group_logp(a, b.frame_arc, i1[v] - 1, total);
        a.o_logp[g] = (float)lp + 0.0f;  // -0.0 and +0.0 compare equal in the reference's sort
      }
    }
  }
  if (!windowed) return;
  __syncthreads();
  const int nlong = min(s_nlong, kLongCap);
  for (int k = threadIdx.x; k < nlong; k += blockDim.x) {
    const int64_t g = row0 + s_long[k];
    const uint32_t i0 = __ldg(a.gstart + g), i1 = __ldg(a.gstart + g + 1);
    double sum = 0.0;
    uint32_t i = i0;
    for (; i + 4 <= i1; i += 4) {  // four ids in flight
      int e[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) e[u] = (int)((unsigned int)__ldg(b.frame_arc + i + u) & 0x7fffffffu) - wlo;
#pragma unroll
      for (int u = 0; u < 4; ++u) sum += s_post[e[u]];
    }
    for (; i < i1; ++i) sum += s_post[(int)((unsigned int)__ldg(b.frame_arc + i) & 0x7fffffffu) - wlo];
    const double lp = sum >= 1e-280 ? fast_log(sum) : exact_group_logp(a, b.frame_arc, i1 - 1, total);
    a.o_logp[g] = (float)lp + 0.0f;
  }
}

// Bitonic sorting network over 32 * R packed 32-bit keys held in registers, R per
// lane, position p = lane * R + r (ascending).  Partners closer than R sit in the same
// lane (two VIMNMX per pair); the others are one shuffle away.
template <int R>
__device__ __forceinline__ void bitonic_regs(unsigned int (&v)[R], int lane) {
  constexpr int N = 32 * R;
#pragma unroll
  for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j < R) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if ((r & j) == 0) {
            const bool up = (k < R) ? ((r & k) == 0) : ((lane & (k / R)) == 0);
            const unsigned int x = v[r], y = v[r | j];
            v[r] = up ? min(x, y) : max(x, y);
            v[r | j] = up ? max(x, y) : min(x, y);
          }
        }
      } else {
        const int m = j / R;
        const bool keep_min = ((lane & (k / R)) == 0) == ((lane & m) == 0);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const unsigned int y = __shfl_xor_sync(0xffffffffu, v[r], m);
          v[r] = keep_min ? min(v[r], y) : max(v[r], y);
        }
      }
    }
  }
}

// Orders the c <= 32 * R rows [dst, dst + c) of frame k by (float logp desc, word asc).
// The network sorts ONE 32-bit word per row: the ordered bits of the log-posterior
// with their lowest log2(32 R) bits replaced by the row's pre-order index (rows are
// stored in ascending word order, so index order = word order).  Rows whose
// log-posteriors agree in all the kept bits can come out in the wrong order; that is
// checked against the full keys afterwards and such a frame (a few per cent) is redone
// with 64-bit keys in shared memory.
template <int R>
__device__ __forceinline__ void order_frame(const FrameArgs& a, int64_t dst, int c, int lane, unsigned int* s_key,
                                            unsigned long long* sortbuf) {
  constexpr unsigned int kMask = 32u * R - 1u;
  unsigned int v[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int e = lane * R + r;
    unsigned int ok = 0xffffffffu, pk = 0xffffffffu;
    if (e < c) {
      ok = ~ord_f32(a.o_logp[dst + e]);
      pk = (ok & ~kMask) | (unsigned int)e;
    }
    s_key[e] = ok;
    v[r] = pk;
  }
  bitonic_regs<R>(v, lane);
  __syncwarp();  // s_key is complete
  // rows leave straight from the registers (position p = lane * R + r); the order is
  // checked against the full keys on the way
  unsigned int fk[R];
#pragma unroll
  for (int r = 0; r < R; ++r) fk[r] = s_key[v[r] & kMask];
  const unsigned int next0 = __shfl_down_sync(0xffffffffu, fk[0], 1);
  bool bad = false;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int p = lane * R + r;
    if (p < c) {
      const unsigned int nx = r + 1 < R ? fk[r + 1 < R ? r + 1 : r] : next0;
      if (p + 1 < c) bad |= fk[r] > nx;
      a.o_word[dst + p] = __ldg(a.gwords + dst + (v[r] & kMask));
      a.o_logp[dst + p] = inv_ord_f32(~fk[r]);
    }
  }
  if (__any_sync(0xffffffffu, bad)) {
    constexpr int N = 32 * R;
    for (int g = lane; g < N; g += 32)
      sortbuf[g] = g < c ? (((unsigned long long)s_key[g] << 32) | (unsigned int)__ldg(a.gwords + dst + g)) : ~0ULL;
    __syncwarp();
    warp_bitonic_fixed<N>(sortbuf, lane);
    for (int g = lane; g < c; g += 32) {
      const unsigned long long sk = sortbuf[g];
      a.o_word[dst + g] = (int32_t)(sk & 0xffffffffu);
      a.o_logp[dst + g] = inv_ord_f32(~(unsigned int)(sk >> 32));
    }
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kFrameWarps * 32, 8) k_frame_order(const __grid_constant__ FrameArgs a) {
  __shared__ __align__(16) unsigned long long s_sort[kFrameWarps][kGroupCap];
  __shared__ unsigned int s_keys[kFrameWarps][kGroupCap];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BatchView& b = a.b;
  for (int item = blockIdx.x * kFrameWarps + warp; item < a.num_items; item += gridDim.x * kFrameWarps) {
    const int l = last_le(a.item_base, 0, b.L - 1, item);  // lattice of this item
    const int T = b.fr_base[l + 1] - b.fr_base[l] - 1;
    const int k0 = (item - a.item_base[l]) * kFramesPerItem;
    const int k1 = min(T, k0 + kFramesPerItem);
    const int64_t* gl = a.gloc + b.fr_base[l];
    const int64_t out0 = a.res_off[l];
    int64_t g_next = gl[k0];
    {
      // the run's rows are two contiguous ranges (log-posteriors, words): ask L2 for them
      // now, the frames below then wait on L2 rather than on HBM, one after the other
      const int64_t nb = (gl[k1] - g_next) * 4;
      const char* q0 = reinterpret_cast<const char*>(a.o_logp + out0 + g_next);
      const char* q1 = reinterpret_cast<const char*>(a.gwords + out0 + g_next);
      for (int64_t off = lane * 128; off < nb; off += 32 * 128) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(q0 + off));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(q1 + off));
      }
    }
    for (int k = k0; k < k1; ++k) {
      const int64_t g0 = g_next;
      g_next = gl[k + 1];
      const int c = (int)(g_next - g0);
      if (c == 0) continue;
      const int64_t dst = out0 + g0;
      if (c <= 32) order_frame<1>(a, dst, c, lane, s_keys[warp], s_sort[warp]);
      else if (c <= 64) order_frame<2>(a, dst, c, lane, s_keys[warp], s_sort[warp]);
      else if (c <= 128) order_frame<4>(a, dst, c, lane, s_keys[warp], s_sort[warp]);
      else if (c <= 256) order_frame<8>(a, dst, c, lane, s_keys[warp], s_sort[warp]);
      else {
        for (int g = lane; g < c; g += 32) a.o_word[dst + g] = __ldg(a.gwords + dst + g);
        __syncwarp();
        warp_sort_rows_global(a.o_logp + dst, a.o_word + dst, c, lane);
      }
    }
  }
}

// ----------------------------------------------------------- pack-time build ---
struct GroupArgs {
  BatchView b;
  int bits_label;
  const int64_t* inst_base;  // [L+1] first instance of each lattice
  unsigned long long* key;   // sort input: (frame << bits_label) | word
  unsigned int* val;         //             out-order arc id
  const unsigned long long *key_a, *key_b;
  const unsigned int *val_a, *val_b;
  const unsigned char* where;
  int k32;                   // the (frame, word) keys fit 32 bits: the key buffers hold unsigned ints
  int32_t* frame_arc;
  int32_t* frame_cnt;        // per frame slot: groups in the frame
  const int32_t* item_base;
  int num_items;
  int64_t* gloc;
  int32_t* lat_cnt;
  const int64_t* res_off;
  int32_t* gwords;
  int32_t* gframe;
  uint32_t* gstart;
  int32_t *run_lo, *run_hi;
  int32_t* max_window;       // largest window of the batch
  const int64_t* arc_base;   // [L] = e_off as 64-bit segment bases
  int32_t* rank_of;          // [E] out-order arc -> time-order index (global)
  int4* tarc;
  int32_t* tlabel;
};

// grid (L, tiles): sort input for the time order: key = start frame, val = out-order arc (lattice-local)
__global__ void __launch_bounds__(256) k_fg_time_keys(GroupArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  for (int e = e0 + lt.tile * blockDim.x + threadIdx.x; e < e1; e += lt.tiles * blockDim.x) {
    reinterpret_cast<unsigned int*>(a.key)[e] = (unsigned int)max(a.b.time[a.b.out_src[e]], 0);  // 32-bit keys
    a.val[e] = (unsigned int)(e - e0);
  }
}

// grid (L, tiles): the time-ordered arc copy and the inverse permutation
__global__ void __launch_bounds__(256) k_fg_time_copy(GroupArgs a) {
  const LatTile lt = lat_tile();  // CTAs that run together share lattices (L2 locality)
  const int l = lt.l;
  const int e0 = a.b.e_off[l], e1 = a.b.e_off[l + 1];
  const unsigned int* val = (a.where[l] ? a.val_b : a.val_a) + e0;
  for (int j = e0 + lt.tile * blockDim.x + threadIdx.x; j < e1; j += lt.tiles * blockDim.x) {
    const int e = e0 + (int)val[j - e0];
    const int4 r = a.b.out_rec[e];
    a.tarc[j] = make_int4(a.b.out_src[e], r.x, r.y, r.z);
    a.tlabel[j] = r.w;
    a.rank_of[e] = j;
  }
}

__device__ __forceinline__ int arc_frames(const BatchView& b, int e, int T, int* first) {
  const int4 r = b.out_rec[e];
  if (r.w == 0) return 0;
  const int fa = max(b.time[b.out_src[e]], 0), fb = min(b.time[r.x], T);
  *first = fa;
  return fb > fa ? fb - fa : 0;
}

// One CTA per lattice: exclusive scan of the arcs' frame counts, then the
// (frame, word) -> arc instances in arc order, each carrying the arc's TIME-ORDER index
// (the stable sort then leaves every group in a fixed order).
__global__ void __launch_bounds__(256) k_fg_emit(GroupArgs a) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = blockIdx.x;
  const BatchView& b = a.b;
  const int e0 = b.e_off[l], e1 = b.e_off[l + 1];
  const int T = b.fr_base[l + 1] - b.fr_base[l] - 1;
  const int64_t base = a.inst_base[l];
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = e0; tile < e1; tile += 256) {
    const int e = tile + tid;
    int first = 0;
    const int cnt = e < e1 ? arc_frames(b, e, T, &first) : 0;
    const int off = cta_exclusive_scan<int, 256>(cnt, warp_sum, carry_s);
    if (cnt > 0) {
      const unsigned long long word = (unsigned long long)(unsigned int)b.out_rec[e].w;
      for (int q = 0; q < cnt; ++q) {
        const unsigned long long k = ((unsigned long long)(first + q) << a.bits_label) | word;
        if (a.k32) reinterpret_cast<unsigned int*>(a.key)[base + off + q] = (unsigned int)k;
        else a.key[base + off + q] = k;
        a.val[base + off + q] = (unsigned int)a.rank_of[e];
      }
    }
  }
}

// one warp per run of frames.  WORDS == false: sorted instances -> frame_arc with head
// bits, groups per frame.  WORDS == true (after the scans): the word of every group,
// in output-row order.
template <bool WORDS>
__global__ void __launch_bounds__(256) k_fg_heads(GroupArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const BatchView& b = a.b;
  for (int item = blockIdx.x * 8 + warp; item < a.num_items; item += gridDim.x * 8) {
    const int l = last_le(a.item_base, 0, b.L - 1, item);
    const int T = b.fr_base[l + 1] - b.fr_base[l] - 1;
    const int k0 = (item - a.item_base[l]) * kFramesPerItem;
    const int k1 = min(T, k0 + kFramesPerItem);
    const unsigned long long* key = a.where[l] ? a.key_b : a.key_a;
    const unsigned int* key32 = reinterpret_cast<const unsigned int*>(key);
    const unsigned int* val = a.where[l] ? a.val_b : a.val_a;
    const unsigned long long label_mask = (1ULL << a.bits_label) - 1ULL;
    int wlo = 0x7fffffff, whi = -1;  // arc id window of the run
    for (int k = k0; k < k1; ++k) {
      const int fs = b.fr_base[l] + k;
      const int64_t f0 = b.fr_off[fs], f1 = b.fr_off[fs + 1];
      int groups = 0;
      for (int64_t i0 = f0; i0 < f1; i0 += 32) {
        const int64_t i = i0 + lane;
        unsigned long long kk = 0;
        bool head = false;
        if (i < f1) {
          kk = a.k32 ? (unsigned long long)key32[i] : key[i];
          head = i == f0 || (a.k32 ? (unsigned long long)key32[i - 1] : key[i - 1]) != kk;
        }
        const unsigned int hm = __ballot_sync(0xffffffffu, head);
        if (!WORDS) {
          if (i < f1) {
            const unsigned int e = val[i];
            a.frame_arc[i] = (int32_t)(e | (head ? 0x80000000u : 0u));
            wlo = min(wlo, (int)e);
            whi = max(whi, (int)e);
          }
        } else if (head) {
          const int64_t row = a.res_off[l] + a.gloc[fs] + groups + __popc(hm & ((1u << lane) - 1u));
          a.gwords[row] = (int32_t)(kk & label_mask);
          a.gframe[row] = k;
          a.gstart[row] = (uint32_t)i;
        }
        groups += __popc(hm);
      }
      if (!WORDS && lane == 0) a.frame_cnt[fs] = groups;
    }
    if (!WORDS) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        wlo = min(wlo, __shfl_xor_sync(0xffffffffu, wlo, o));
        whi = max(whi, __shfl_xor_sync(0xffffffffu, whi, o));
      }
      if (lane == 0) {
        a.run_lo[item] = wlo;
        a.run_hi[item] = whi;
        if (whi >= wlo) atomicMax(a.max_window, whi - wlo + 1);
      }
    }
  }
}

// One CTA per lattice: scan the per-frame group counts into lattice-local output
// rows (T + 1 entries: the last one is the lattice's row count).
__global__ void __launch_bounds__(256) k_fg_scan(GroupArgs a) {
  __shared__ int warp_sum[8];
  __shared__ long long carry_s;
  const int l = blockIdx.x;
  const int f0 = a.b.fr_base[l], T = a.b.fr_base[l + 1] - f0 - 1;
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int tile = 0; tile < T; tile += 256) {
    const int k = tile + tid;
    const int c = k < T ? a.frame_cnt[f0 + k] : 0;
    const long long pre = cta_exclusive_scan<int, 256, long long>(c, warp_sum, carry_s);
    if (k < T) a.gloc[f0 + k] = pre;
  }
  if (tid == 0) {
    a.gloc[f0 + T] = carry_s;
    a.lat_cnt[l] = (int32_t)carry_s;
  }
}

int bits_for(int64_t maxv) {
  int b = 1;
  while (b < 63 && ((int64_t)1 << b) <= maxv) ++b;
  return b;
}

}  // namespace

// Called by both packers once the packed arrays, state times and the frame CSR
// offsets (fr_base, fr_off) are on the device.
int build_frame_groups(klu_ctx* c) {
  const int32_t L = c->L;
  c->h_frame_res_off.assign(L + 1, 0);
  c->fr_items = 0;
  if (L == 0) return 0;
  bool any_bad_times = false;
  for (int32_t l = 0; l < L; ++l) any_bad_times |= !c->h_times_ok[l];
  const int64_t N = c->frame_entries;
  const int64_t F = c->h_fr_base[L];
  std::vector<int32_t> item_base(L + 1, 0);
  std::vector<int64_t> inst_base(L + 1, 0);
  std::vector<int32_t> inst_cnt(L, 0);
  for (int32_t l = 0; l < L; ++l) {
    item_base[l + 1] = item_base[l] + (c->h_num_frames[l] + kFramesPerItem - 1) / kFramesPerItem;
    inst_base[l + 1] = inst_base[l] + c->h_cap_frame[l];
    if (c->h_cap_frame[l] >= ((int64_t)1 << 31)) {
      set_error("lattice " + std::to_string(l) + ": more than 2^31 arc x frame instances");
      return 1;
    }
    inst_cnt[l] = (int32_t)c->h_cap_frame[l];
  }
  c->fr_items = item_base[L];
  KLU_TRY(c->d_fr_item.reserve(4 * (size_t)(L + 1)));
  KLU_TRY(c->d_fr_gloc.reserve(8 * (size_t)std::max<int64_t>(F, 1)));
  KLU_TRY(c->d_fr_res_off.reserve(8 * (size_t)(L + 1)));
  KLU_TRY(small_h2d(c, c->d_fr_item.p, item_base.data(), 4 * (size_t)(L + 1)));
  KLU_CUDA(cudaMemsetAsync(c->d_fr_gloc.p, 0, 8 * (size_t)std::max<int64_t>(F, 1), c->stream));
  KLU_CUDA(cudaMemsetAsync(c->d_fr_res_off.p, 0, 8 * (size_t)(L + 1), c->stream));
  if (N == 0 || any_bad_times) {  // nothing to index (run_frame_post rejects inconsistent times)
    KLU_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  }
  const int bits_label = bits_for(c->max_label), bits_time = bits_for(c->max_time);
  if (N >= ((int64_t)1 << 32) - 1) {
    set_error("klu_load: more than 2^32 arc x frame instances in one batch; split it");
    return 1;
  }
  if (bits_label + bits_time > 62) {
    set_error("frame index key does not fit 62 bits (labels/times too large)");
    return 1;
  }
  // scratch: the context's tool-scratch slots (free while loading; they stay allocated, so
  // repeated loads do not go through cudaMalloc / cudaFree again)
  DevBuf &key_a = c->d_scratch[6], &key_b = c->d_scratch[7], &val_a = c->d_scratch[8], &val_b = c->d_scratch[9],
         &misc = c->d_scratch[10];
  int rc = 0;
  do {
    if ((rc = key_a.reserve(8 * (size_t)N)) || (rc = key_b.reserve(8 * (size_t)N)) ||
        (rc = val_a.reserve(4 * (size_t)N)) || (rc = val_b.reserve(4 * (size_t)N)) ||
        (rc = misc.reserve(8 * (size_t)(L + 1) + 4 * (size_t)L + 4 * (size_t)L + (size_t)L + 4 * (size_t)F + 256)))
      break;
    char* mp = misc.as<char>();
    int64_t* d_inst_base = reinterpret_cast<int64_t*>(mp);
    int32_t* d_inst_cnt = reinterpret_cast<int32_t*>(mp + 8 * (size_t)(L + 1));
    int32_t* d_lat_cnt = d_inst_cnt + L;
    int32_t* d_frame_cnt = d_lat_cnt + L;
    unsigned char* d_where = reinterpret_cast<unsigned char*>(d_frame_cnt + F);
    if ((rc = small_h2d(c, d_inst_base, inst_base.data(), 8 * (size_t)(L + 1)))) break;
    if ((rc = small_h2d(c, d_inst_cnt, inst_cnt.data(), 4 * (size_t)L))) break;
    cudaMemsetAsync(d_frame_cnt, 0, 4 * (size_t)F, c->stream);
    if ((rc = c->d_frame_arc.reserve(4 * (size_t)N))) break;
    GroupArgs a;
    a.b = c->view();
    a.bits_label = bits_label;
    a.inst_base = d_inst_base;
    a.key = key_a.as<unsigned long long>();
    a.val = val_a.as<unsigned int>();
    a.key_a = key_a.as<unsigned long long>();
    a.key_b = key_b.as<unsigned long long>();
    a.val_a = val_a.as<unsigned int>();
    a.val_b = val_b.as<unsigned int>();
    a.where = d_where;
    a.frame_arc = c->d_frame_arc.as<int32_t>();
    a.frame_cnt = d_frame_cnt;
    a.item_base = c->d_fr_item.as<int32_t>();
    a.num_items = c->fr_items;
    a.gloc = c->d_fr_gloc.as<int64_t>();
    a.lat_cnt = d_lat_cnt;
    // ---- arcs by start time: a copy the frame kernels index (a run of frames then touches
    //      one contiguous range of it), and the out-order -> time-order map for the instances
    {
      const size_t E1 = (size_t)std::max<int64_t>(c->E, 1);
      if ((rc = key_a.reserve(8 * std::max<size_t>((size_t)N, E1))) || (rc = key_b.reserve(8 * std::max<size_t>((size_t)N, E1))) ||
          (rc = val_a.reserve(4 * std::max<size_t>((size_t)N, E1))) || (rc = val_b.reserve(4 * std::max<size_t>((size_t)N, E1))) ||
          (rc = c->d_scratch[11].reserve(4 * E1)) || (rc = c->d_fr_tarc.reserve(16 * E1)) ||
          (rc = c->d_fr_tlabel.reserve(4 * E1)))
        break;
      a.key = key_a.as<unsigned long long>();
      a.val = val_a.as<unsigned int>();
      a.key_a = key_a.as<unsigned long long>();
      a.key_b = key_b.as<unsigned long long>();
      a.val_a = val_a.as<unsigned int>();
      a.val_b = val_b.as<unsigned int>();
      a.rank_of = c->d_scratch[11].as<int32_t>();
      a.tarc = c->d_fr_tarc.as<int4>();
      a.tlabel = c->d_fr_tlabel.as<int32_t>();
      int64_t max_arcs = 0;
      std::vector<int64_t> arc_base(L + 1);
      std::vector<int32_t> arc_cnt(L);
      for (int32_t l = 0; l < L; ++l) {
        max_arcs = std::max(max_arcs, c->h_e_off[l + 1] - c->h_e_off[l]);
        arc_base[l] = c->h_e_off[l];
        arc_cnt[l] = (int32_t)(c->h_e_off[l + 1] - c->h_e_off[l]);
      }
      arc_base[L] = c->h_e_off[L];
      const int arc_tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
      DevBuf& seg = c->d_fr_seg;  // persistent: a cudaFree here would stall the other contexts of the device
      if ((rc = seg.reserve(8 * (size_t)(L + 1) + 4 * (size_t)L))) break;
      if ((rc = small_h2d(c, seg.p, arc_base.data(), 8 * (size_t)(L + 1)))) break;
      if ((rc = small_h2d(c, seg.as<char>() + 8 * (size_t)(L + 1), arc_cnt.data(), 4 * (size_t)L))) break;
      {
        KLU_LAUNCH(c, "k_fg_time_keys");
        k_fg_time_keys<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a);
      }
      rc = check_launch("k_fg_time_keys");
      if (!rc) {
        SegSortArgs32 st;  // frame numbers: one 10-bit pass at T <= 1023
        st.seg_base = seg.as<int64_t>();
        st.seg_cnt = reinterpret_cast<const int32_t*>(seg.as<char>() + 8 * (size_t)(L + 1));
        st.key_a = key_a.as<unsigned int>();
        st.val_a = val_a.as<unsigned int>();
        st.key_b = key_b.as<unsigned int>();
        st.val_b = val_b.as<unsigned int>();
        st.where = d_where;
        st.lo_bit = 0;
        st.hi_bit = bits_time;
        {
          KLU_LAUNCH(c, "k_seg_radix_sort");
          rc = seg_sort_launch(c, st, L, c->E);
        }
        if (!rc) rc = check_launch("k_seg_radix_sort(arc start times)");
      }
      if (!rc) {
        KLU_LAUNCH(c, "k_fg_time_copy");
        k_fg_time_copy<<<dim3(L, arc_tiles), 256, 0, c->stream>>>(a);
        rc = check_launch("k_fg_time_copy");
      }
      cudaStreamSynchronize(c->stream);  // arc_base / arc_cnt go out of scope
      if (rc) break;
    }
    a.k32 = bits_label + bits_time <= 32 ? 1 : 0;
    {
      KLU_LAUNCH(c, "k_fg_emit");
      k_fg_emit<<<L, 256, 0, c->stream>>>(a);
    }
    if ((rc = check_launch("k_fg_emit"))) break;
    if (a.k32) {  // (frame, word) fits 32 bits: a third less traffic per pass
      SegSortArgs32 ss;
      ss.seg_base = d_inst_base;
      ss.seg_cnt = d_inst_cnt;
      ss.key_a = key_a.as<unsigned int>();
      ss.val_a = val_a.as<unsigned int>();
      ss.key_b = key_b.as<unsigned int>();
      ss.val_b = val_b.as<unsigned int>();
      ss.where = d_where;
      ss.lo_bit = 0;
      ss.hi_bit = bits_label + bits_time;
      KLU_LAUNCH(c, "k_seg_radix_sort");
      if ((rc = seg_sort_launch(c, ss, L, N))) break;
    } else {
      SegSortArgs ss;
      ss.seg_base = d_inst_base;
      ss.seg_cnt = d_inst_cnt;
      ss.key_a = key_a.as<unsigned long long>();
      ss.val_a = val_a.as<unsigned int>();
      ss.key_b = key_b.as<unsigned long long>();
      ss.val_b = val_b.as<unsigned int>();
      ss.where = d_where;
      ss.lo_bit = 0;
      ss.hi_bit = bits_label + bits_time;
      KLU_LAUNCH(c, "k_seg_radix_sort");
      if ((rc = seg_sort_launch(c, ss, L, N))) break;
    }
    if ((rc = check_launch("k_seg_radix_sort(frame groups)"))) break;
    a.res_off = c->d_fr_res_off.as<int64_t>();
    a.gwords = nullptr;
    if ((rc = c->d_fr_run_lo.reserve(4 * (size_t)std::max(a.num_items, 1)))) break;
    if ((rc = c->d_fr_run_hi.reserve(4 * (size_t)std::max(a.num_items, 1)))) break;
    a.run_lo = c->d_fr_run_lo.as<int32_t>();
    a.run_hi = c->d_fr_run_hi.as<int32_t>();
    a.max_window = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(d_where) + (((size_t)L + 3) & ~(size_t)3));  // spare int of the misc block
    cudaMemsetAsync(a.max_window, 0, 4, c->stream);
    const int hgrid = std::max(1, std::min((a.num_items + 7) / 8, c->num_sms * 32));
    if (a.num_items > 0) {
      KLU_LAUNCH(c, "k_fg_heads");
      k_fg_heads<false><<<hgrid, 256, 0, c->stream>>>(a);
    }
    if ((rc = check_launch("k_fg_heads"))) break;
    {
      KLU_LAUNCH(c, "k_fg_scan");
      k_fg_scan<<<L, 256, 0, c->stream>>>(a);
    }
    if ((rc = check_launch("k_fg_scan"))) break;
    if ((rc = scan_counts(c, d_lat_cnt, 0, L, c->d_fr_res_off.as<int64_t>(), "k_fg_latscan"))) break;
    if ((rc = small_d2h(c, &c->fr_max_window, a.max_window, 4))) break;
    if ((rc = small_d2h(c, c->h_frame_res_off.data(), c->d_fr_res_off.p, 8 * (size_t)(L + 1)))) break;
    if ((rc = small_sync(c))) break;
    if ((rc = c->d_fr_gword.reserve(4 * (size_t)std::max<int64_t>(c->h_frame_res_off[L], 1)))) break;
    if ((rc = c->d_fr_gstart.reserve(4 * (size_t)(c->h_frame_res_off[L] + 1)))) break;
    if ((rc = c->d_fr_gframe.reserve(4 * (size_t)std::max<int64_t>(c->h_frame_res_off[L], 1)))) break;
    a.gwords = c->d_fr_gword.as<int32_t>();
    a.gframe = c->d_fr_gframe.as<int32_t>();
    a.gstart = c->d_fr_gstart.as<uint32_t>();
    {
      const uint32_t n32 = (uint32_t)N;
      if ((rc = small_h2d(c, a.gstart + c->h_frame_res_off[L], &n32, 4))) break;
    }
    if (a.num_items > 0) {
      KLU_LAUNCH(c, "k_fg_words");
      k_fg_heads<true><<<hgrid, 256, 0, c->stream>>>(a);
    }
    if ((rc = check_launch("k_fg_words"))) break;
  } while (0);
  cudaStreamSynchronize(c->stream);
  return rc;
}

int run_frame_post(klu_ctx* c, const klu_opts* o) {
  const int32_t L = c->L;
  KLU_TRY(ensure_frame_index(c));
  for (int32_t l = 0; l < L; ++l)
    if (!c->h_times_ok[l]) {
      set_error("lattice " + std::to_string(l) + ": inconsistent state times (lattice is not aligned)");
      return 1;
    }
  CostParams cp = make_cost_params(o, false);
  KLU_TRY(run_log_sweeps(c, cp, false, 0.f));
  c->h_res_off = c->h_frame_res_off;
  c->frame_col_static = true;
  c->h_res_off.resize(L + 1, 0);
  c->last_entries = L ? c->h_res_off[L] : 0;
  if (L == 0) return 0;
  const int64_t N = std::max<int64_t>(c->last_entries, 1);
  KLU_TRY(c->d_res[5].reserve(8 * (size_t)(L + 1)));
  KLU_TRY(c->d_res[1].reserve(4 * (size_t)N));
  KLU_TRY(c->d_res[4].reserve(4 * (size_t)N));
  KLU_CUDA(cudaMemcpyAsync(c->d_res[5].p, c->d_fr_res_off.p, 8 * (size_t)(L + 1), cudaMemcpyDeviceToDevice, c->stream));
  if (c->last_entries == 0) return 0;
  FrameArgs a;
  a.b = c->view();
  a.cp = make_cost_params(o, true);  // the arc term is (float)(g + a)
  a.alpha = c->d_alpha.as<double>();
  a.beta = c->d_beta.as<double>();
  a.total = c->d_total.as<double>();
  a.item_base = c->d_fr_item.as<int32_t>();
  a.num_items = c->fr_items;
  a.gloc = c->d_fr_gloc.as<int64_t>();
  a.res_off = c->d_fr_res_off.as<int64_t>();
  a.gwords = c->d_fr_gword.as<int32_t>();
  a.gstart = c->d_fr_gstart.as<uint32_t>();
  a.o_word = c->d_res[1].as<int32_t>();
  a.o_logp = c->d_res[4].as<float>();
  a.run_lo = c->d_fr_run_lo.as<int32_t>();
  a.run_hi = c->d_fr_run_hi.as<int32_t>();
  a.tarc = c->d_fr_tarc.as<int4>();
  a.tlabel = c->d_fr_tlabel.as<int32_t>();
  if (a.num_items > 0) {
    // shared memory: the largest window of the batch, capped (runs beyond the cap take the slow path)
    const int kMaxWinBytes = 64 << 10;
    KLU_CUDA(cudaFuncSetAttribute(k_frame_groups, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxWinBytes));  // per device
    const int kWinBytes = std::min(kMaxWinBytes, std::max(1024, (c->fr_max_window * 8 + 1023) & ~1023));
    a.win_cap = kWinBytes / 8;
    KLU_LAUNCH(c, "k_frame_groups");
    k_frame_groups<<<a.num_items, 128, kWinBytes, c->stream>>>(a);
    KLU_TRY(check_launch("k_frame_groups"));
  }
  if (a.num_items > 0) {
    const int grid = std::max(1, std::min((a.num_items + kFrameWarps - 1) / kFrameWarps, c->num_sms * 64));
    {
      KLU_LAUNCH(c, "k_frame_order");
      k_frame_order<<<grid, kFrameWarps * 32, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_frame_order"));
  }
  return 0;
}

}  // namespace klu
