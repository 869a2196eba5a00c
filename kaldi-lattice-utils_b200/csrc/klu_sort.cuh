// klu_sort.cuh -- batched segmented LSD radix sort (SURVEY.md K7/K8 building block).
//
// One CTA sorts one segment (one lattice's index entries) of (u64 key, u32 value)
// pairs, stable, 8 bits per pass, ping-ponging between two global buffers.  All
// digit histograms are taken in ONE read of the keys; passes whose digit is the
// same for every key of the segment are skipped, so keys may be laid out
// generously.  where[l] tells the consumer which buffer holds segment l.
#pragma once
#include <stdlib.h>

#include <algorithm>

#include "klu_common.cuh"

namespace klu {

constexpr int kSortItems = 4;

template <typename K>
struct SegSortArgsT {
  const int64_t* seg_base;  // [nseg] first element of each segment
  const int32_t* seg_cnt;   // [nseg] elements in each segment
  K* key_a;
  unsigned int* val_a;
  K* key_b;
  unsigned int* val_b;
  unsigned char* where;  // [nseg] out: 0 = result in a, 1 = result in b
  int lo_bit, hi_bit;
};
typedef SegSortArgsT<unsigned long long> SegSortArgs;
typedef SegSortArgsT<unsigned int> SegSortArgs32;  // 32-bit keys: a third less traffic per pass

#ifdef __CUDACC__
// Lanes of the warp whose (valid) element has the same 8-bit digit: eight ballots, constant cost.
// (__match_any_sync does the same in one instruction but its cost grows with the number of
// distinct values: on the random low digits of the order keys it was the bottleneck of the
// ranking -- ncu: short-scoreboard / MIO stalls, 10-16 % of the issue slots used.)
static __device__ __forceinline__ unsigned int match_digit(int d, bool valid) {
  unsigned int m = __ballot_sync(0xffffffffu, valid);
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const bool bit = (d >> b) & 1;
    const unsigned int bal = __ballot_sync(0xffffffffu, bit);
    m &= bit ? bal : ~bal;
  }
  return m;
}

// BITS = digit width (8, 9 or 10): 26-bit (frame, word) keys take three 9-bit passes instead of
// four 8-bit ones, 10-bit frame numbers one pass instead of two (seg_sort_launch picks the width).
constexpr int kSortThreads = 512;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortTile = kSortThreads * kSortItems;

template <int BITS>
static __device__ __forceinline__ unsigned int match_digit_w(int d, bool valid) {
  unsigned int m = __ballot_sync(0xffffffffu, valid);
#pragma unroll
  for (int b = 0; b < BITS; ++b) {
    const bool bit = (d >> b) & 1;
    const unsigned int bal = __ballot_sync(0xffffffffu, bit);
    m &= bit ? bal : ~bal;
  }
  return m;
}

template <typename K, int BITS>
static __global__ void __launch_bounds__(kSortThreads) k_seg_radix_sort_t(SegSortArgsT<K> a) {
  constexpr int NB = 1 << BITS;
  constexpr int PER = NB > kSortThreads ? NB / kSortThreads : 1;  // bins per thread in the bin scan
  extern __shared__ unsigned int sort_smem[];
  __shared__ unsigned int wsum[kSortWarps];
  __shared__ int skip_flag;
  const int seg = blockIdx.x;
  const int n = a.seg_cnt[seg];
  const int64_t base = a.seg_base[seg];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int npass = (a.hi_bit - a.lo_bit + BITS - 1) / BITS;
  if (n <= 1 || npass <= 0) {
    if (tid == 0) a.where[seg] = 0;
    return;
  }
  unsigned int* bin_base = sort_smem;                                  // [NB]
  unsigned int(*warp_cnt)[NB] = reinterpret_cast<unsigned int(*)[NB]>(sort_smem + NB);  // [kSortWarps][NB]
  unsigned int(*hist)[NB] = reinterpret_cast<unsigned int(*)[NB]>(sort_smem + NB + kSortWarps * NB);  // [npass][NB]
  K* kin = a.key_a + base;
  unsigned int* vin = a.val_a + base;
  K* kout = a.key_b + base;
  unsigned int* vout = a.val_b + base;
  for (int i = tid; i < npass * NB; i += kSortThreads) (&hist[0][0])[i] = 0;
  __syncthreads();
  for (int i0 = 0; i0 < n; i0 += 4 * kSortThreads) {
    K kk[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {  // four requests in flight per thread
      const int i = i0 + r * kSortThreads + tid;
      kk[r] = i < n ? kin[i] : (K)0;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (i0 + r * kSortThreads + tid >= n) break;
      const K k = kk[r] >> a.lo_bit;
      for (int p = 0; p < npass; ++p) atomicAdd(&hist[p][(unsigned int)(k >> (BITS * p)) & (unsigned int)(NB - 1)], 1u);
    }
  }
  __syncthreads();
  int executed = 0;
  for (int p = 0; p < npass; ++p) {
    const int shift = a.lo_bit + BITS * p;
    if (tid == 0) skip_flag = 0;
    __syncthreads();
    for (int b = tid; b < NB; b += kSortThreads)
      if (hist[p][b] == (unsigned)n) skip_flag = 1;
    __syncthreads();
    if (skip_flag) continue;
    // exclusive scan of hist[p] -> bin_base: thread t owns bins [t * PER, (t + 1) * PER)
    {
      unsigned int mine[PER];
      unsigned int tot = 0;
#pragma unroll
      for (int q = 0; q < PER; ++q) {
        const int b = tid * PER + q;
        mine[q] = b < NB ? hist[p][b] : 0u;
        tot += mine[q];
      }
      unsigned int x = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) wsum[warp] = x;
      __syncthreads();
      unsigned int run = x - tot;
      for (int w = 0; w < warp; ++w) run += wsum[w];
#pragma unroll
      for (int q = 0; q < PER; ++q) {
        const int b = tid * PER + q;
        if (b < NB) bin_base[b] = run;
        run += mine[q];
      }
    }
    __syncthreads();
    // The loads of a tile are issued together (kSortItems independent requests per thread) and
    // one tile ahead: the next tile's keys travel while this one is ranked and scattered.
    K k[kSortItems], kn[kSortItems];
    unsigned int v[kSortItems], vn[kSortItems];
#pragma unroll
    for (int r = 0; r < kSortItems; ++r) {
      const int i = (warp * kSortItems + r) * 32 + lane;
      k[r] = i < n ? kin[i] : (K)0;
      v[r] = i < n ? vin[i] : 0u;
    }
    for (int tile = 0; tile < n; tile += kSortTile) {
      for (int i = lane; i < NB; i += 32) warp_cnt[warp][i] = 0;
      __syncwarp();
      int d[kSortItems];
      unsigned int mk[kSortItems];
#pragma unroll
      for (int r = 0; r < kSortItems; ++r) {
        const int i = tile + (warp * kSortItems + r) * 32 + lane;
        const bool valid = i < n;
        d[r] = valid ? (int)((k[r] >> shift) & (K)(NB - 1)) : 0;
        mk[r] = match_digit_w<BITS>(d[r], valid);
        if (valid && lane == __ffs(mk[r]) - 1) warp_cnt[warp][d[r]] += __popc(mk[r]);
        __syncwarp();
      }
#pragma unroll
      for (int r = 0; r < kSortItems; ++r) {
        const int i = tile + kSortTile + (warp * kSortItems + r) * 32 + lane;
        kn[r] = i < n ? kin[i] : (K)0;
        vn[r] = i < n ? vin[i] : 0u;
      }
      __syncthreads();
      for (int b = tid; b < NB; b += kSortThreads) {
        unsigned int run = bin_base[b];
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) {
          const unsigned int cnt = warp_cnt[w][b];
          warp_cnt[w][b] = run;
          run += cnt;
        }
        bin_base[b] = run;
      }
      __syncthreads();
#pragma unroll
      for (int r = 0; r < kSortItems; ++r) {
        const int i = tile + (warp * kSortItems + r) * 32 + lane;
        const bool valid = i < n;
        const unsigned int mask = mk[r];
        const int leader = valid ? __ffs(mask) - 1 : lane;
        unsigned int pos = 0;
        if (valid && lane == leader) {
          pos = warp_cnt[warp][d[r]];
          warp_cnt[warp][d[r]] = pos + __popc(mask);
        }
        pos = __shfl_sync(0xffffffffu, pos, leader);
        if (valid) {
          const unsigned int dst = pos + __popc(mask & ((1u << lane) - 1u));
          kout[dst] = k[r];
          vout[dst] = v[r];
        }
        __syncwarp();
      }
      __syncthreads();
#pragma unroll
      for (int r = 0; r < kSortItems; ++r) {
        k[r] = kn[r];
        v[r] = vn[r];
      }
    }
    // swap buffers
    K* tk = kin;
    kin = kout;
    kout = tk;
    unsigned int* tv = vin;
    vin = vout;
    vout = tv;
    ++executed;
    __syncthreads();
  }
  if (tid == 0) a.where[seg] = (unsigned char)(executed & 1);
}

// digit width: 8 bits unless 9 or 10 save a pass (keys of at most 30 bits: the wider histograms
// live in shared memory per pass)
static inline int seg_sort_digit_bits(int bits) {
  if (bits <= 0 || bits > 30) return 8;
  const int np8 = (bits + 7) / 8, np9 = (bits + 8) / 9, np10 = (bits + 9) / 10;
  if (np9 < np8) return 9;
  if (np10 < np8) return 10;
  return 8;
}

template <typename K, int BITS>
static inline void seg_sort_launch_w(const SegSortArgsT<K>& a, int nseg, cudaStream_t stream) {
  const int npass = (a.hi_bit - a.lo_bit + BITS - 1) / BITS;
  const size_t smem = (size_t)(1 + kSortWarps + std::max(npass, 1)) * (1u << BITS) * 4;
  cudaFuncSetAttribute(k_seg_radix_sort_t<K, BITS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  // per device
  k_seg_radix_sort_t<K, BITS><<<nseg, kSortThreads, smem, stream>>>(a);
}

template <typename K>
static inline void seg_sort_launch(const SegSortArgsT<K>& a, int nseg, cudaStream_t stream) {
  if (nseg <= 0) return;
  const int w = seg_sort_digit_bits(a.hi_bit - a.lo_bit);
  if (w == 9) seg_sort_launch_w<K, 9>(a, nseg, stream);
  else if (w == 10) seg_sort_launch_w<K, 10>(a, nseg, stream);
  else seg_sort_launch_w<K, 8>(a, nseg, stream);
}

// ---------------------------------------------------------------------------------------------
// The same sort with SEVERAL CTAs per segment, for batches of few, large segments (the order
// sort of lattice-word-index-position: a few hundred lattices x ~1.6 M cells; the candidate
// sorts of the character tools: 64 lattices x up to 2^24 candidates) where one CTA per segment
// leaves most of the SMs idle.  Classic three-kernel LSD pass over tiles of kMsTile elements:
//   k_ms_count    per tile: histogram of the pass's digit           -> counts[tile][256]
//   k_ms_scan     per segment: exclusive scan over (digit, tile)    -> first output slot of
//                 every (tile, digit); detects a digit shared by the whole segment (pass skipped)
//   k_ms_scatter  per tile: stable ranks inside the tile + the slot -> the other buffer
// Tiles are cut per segment (segment l owns tiles [tile_first[l], tile_first[l+1])); the
// count / scatter kernels are persistent over the tile list, which stays on the device.
constexpr int kMsThreads = 512;
constexpr int kMsItems = 8;
constexpr int kMsWarps = kMsThreads / 32;
constexpr int kMsTile = kMsThreads * kMsItems;

struct MsWork {
  int32_t* tile_first;      // [nseg + 1]
  int32_t* tile_seg;        // [tiles] segment of every tile
  unsigned int* counts;     // [tiles][256]
  unsigned char* where_in;  // [nseg] buffer holding each segment before this pass
  unsigned char* where_out; // [nseg] ... after it
  unsigned char* skip;      // [nseg] pass skipped for the segment
  int nseg;
};

static __global__ void __launch_bounds__(1024) k_ms_plan(const int32_t* seg_cnt, int nseg, int32_t* tile_first) {
  __shared__ int warp_sum[32];
  __shared__ int carry_s;
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < nseg; base += 1024) {
    const int i = base + tid;
    const int n = i < nseg ? seg_cnt[i] : 0;
    const int c = n <= 1 ? 0 : (n + kMsTile - 1) / kMsTile;
    const int pre = cta_exclusive_scan<int, 1024>(c, warp_sum, carry_s);
    if (i < nseg) tile_first[i] = pre;
  }
  if (tid == 0) tile_first[nseg] = carry_s;
}

static __global__ void __launch_bounds__(256) k_ms_tilemap(MsWork w) {
  const int seg = blockIdx.x;
  for (int t = w.tile_first[seg] + threadIdx.x; t < w.tile_first[seg + 1]; t += blockDim.x) w.tile_seg[t] = seg;
}

// What a CTA needs to know about a tile; fetched one tile ahead so the dependent loads
// (tile -> segment -> its size / base / buffer) are off the critical path.
struct MsTile {
  int seg, n, tile0;
  int64_t base;
  int in_b, skip;
};
template <typename K>
static __device__ __forceinline__ MsTile ms_tile(const SegSortArgsT<K>& a, const MsWork& w, int t, int T, bool want_skip) {
  MsTile x;
  x.seg = -1;
  x.n = 0;
  x.tile0 = 0;
  x.base = 0;
  x.in_b = 0;
  x.skip = 0;
  if (t < T) {
    x.seg = w.tile_seg[t];
    x.n = a.seg_cnt[x.seg];
    x.base = a.seg_base[x.seg];
    x.in_b = w.where_in[x.seg];
    x.tile0 = (t - w.tile_first[x.seg]) * kMsTile;
    x.skip = want_skip ? w.skip[x.seg] : 0;
  }
  return x;
}

template <typename K>
static __global__ void __launch_bounds__(kMsThreads) k_ms_count(SegSortArgsT<K> a, MsWork w, int shift) {
  __shared__ unsigned int hist[256];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = w.tile_first[w.nseg];
  MsTile nx = ms_tile(a, w, blockIdx.x, T, false);
  for (int t = blockIdx.x; t < T; t += gridDim.x) {
    const MsTile cur = nx;
    nx = ms_tile(a, w, t + gridDim.x, T, false);
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    const int n = cur.n;
    const K* kin = (cur.in_b ? a.key_b : a.key_a) + cur.base;
    K k[kMsItems];
#pragma unroll
    for (int r = 0; r < kMsItems; ++r) {
      const int i = cur.tile0 + (warp * kMsItems + r) * 32 + lane;
      k[r] = i < n ? kin[i] : (K)0;
    }
#pragma unroll
    for (int r = 0; r < kMsItems; ++r) {
      const int i = cur.tile0 + (warp * kMsItems + r) * 32 + lane;
      const bool valid = i < n;
      const int d = valid ? (int)((k[r] >> shift) & 255) : -1;
      int same;
      __match_all_sync(0xffffffffu, d, &same);
      if (same) {  // the whole warp has one digit (constant high bytes): one add
        if (lane == 0 && valid) atomicAdd(&hist[d], 32u);
      } else if (valid) {
        atomicAdd(&hist[d], 1u);
      }
    }
    __syncthreads();
    if (tid < 256) w.counts[(size_t)t * 256 + tid] = hist[tid];
    __syncthreads();
  }
}

// one CTA of 256 threads per segment; thread d walks the segment's tiles
static __global__ void __launch_bounds__(256) k_ms_scan(const int32_t* seg_cnt, MsWork w) {
  __shared__ unsigned int tot[256];
  __shared__ unsigned int wsum[8];
  __shared__ int skip_s;
  const int seg = blockIdx.x, d = threadIdx.x, lane = d & 31, warp = d >> 5;
  const int t0 = w.tile_first[seg], t1 = w.tile_first[seg + 1];
  const unsigned int n = (unsigned int)seg_cnt[seg];
  if (d == 0) skip_s = t0 == t1 ? 1 : 0;
  __syncthreads();
  unsigned int run = 0;
  for (int t = t0; t < t1; t += 8) {  // eight independent loads in flight
    unsigned int cc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) cc[q] = t + q < t1 ? w.counts[(size_t)(t + q) * 256 + d] : 0u;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (t + q < t1) w.counts[(size_t)(t + q) * 256 + d] = run;
      run += cc[q];
    }
  }
  if (t1 > t0 && run == n) skip_s = 1;  // every key of the segment has this digit
  // exclusive scan of the digit totals
  unsigned int x = run;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) wsum[warp] = x;
  __syncthreads();
  unsigned int add = 0;
  for (int q = 0; q < warp; ++q) add += wsum[q];
  tot[d] = add + x - run;
  const int skip = skip_s;
  if (d == 0) {
    w.skip[seg] = (unsigned char)skip;
    w.where_out[seg] = (unsigned char)(w.where_in[seg] ^ (skip ? 0 : 1));
  }
  if (skip) return;
  const unsigned int base = tot[d];
  if (base)
    for (int t = t0; t < t1; t += 8) {
      unsigned int cc[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) cc[q] = t + q < t1 ? w.counts[(size_t)(t + q) * 256 + d] : 0u;
#pragma unroll
      for (int q = 0; q < 8; ++q)
        if (t + q < t1) w.counts[(size_t)(t + q) * 256 + d] = cc[q] + base;
    }
}

// The tile is put in digit order in shared memory first, so the stores to the other buffer go out
// as runs of consecutive elements (a warp store touches ~2-4 sectors instead of up to 32: the
// uncoalesced 4-byte scatter was bound by L2 sector writes, not by HBM).
template <typename K>
static __global__ void __launch_bounds__(kMsThreads) k_ms_scatter(SegSortArgsT<K> a, MsWork w, int shift) {
  extern __shared__ unsigned long long ms_smem[];
  K* s_key = reinterpret_cast<K*>(ms_smem);                                  // [kMsTile]
  unsigned int* s_val = reinterpret_cast<unsigned int*>(s_key + kMsTile);    // [kMsTile]
  unsigned int(*warp_cnt)[256] = reinterpret_cast<unsigned int(*)[256]>(s_val + kMsTile);  // [kMsWarps][256]
  unsigned int* tile_prefix = &warp_cnt[0][0] + kMsWarps * 256;              // [256] first tile-local slot of a digit
  unsigned int* gfirst = tile_prefix + 256;                                  // [256] first global slot of a digit
  unsigned int* wsum = gfirst + 256;                                         // [8]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = w.tile_first[w.nseg];
  MsTile nx = ms_tile(a, w, blockIdx.x, T, true);
  for (int t = blockIdx.x; t < T; t += gridDim.x) {
    const MsTile cur = nx;
    nx = ms_tile(a, w, t + gridDim.x, T, true);
    if (cur.skip) continue;  // uniform over the CTA
    for (int i = lane; i < 256; i += 32) warp_cnt[warp][i] = 0;
    __syncwarp();
    const int n = cur.n;
    const bool in_b = cur.in_b != 0;
    const K* kin = (in_b ? a.key_b : a.key_a) + cur.base;
    const unsigned int* vin = (in_b ? a.val_b : a.val_a) + cur.base;
    K* kout = (in_b ? a.key_a : a.key_b) + cur.base;
    unsigned int* vout = (in_b ? a.val_a : a.val_b) + cur.base;
    const int tile0 = cur.tile0;
    const int tile_n = min(kMsTile, n - tile0);
    const unsigned int first_slot = tid < 256 ? w.counts[(size_t)t * 256 + tid] : 0u;  // early: used after the ranking
    K k[kMsItems];
    unsigned int v[kMsItems], mk[kMsItems];
    int d[kMsItems];
#pragma unroll
    for (int r = 0; r < kMsItems; ++r) {
      const int i = tile0 + (warp * kMsItems + r) * 32 + lane;
      k[r] = i < n ? kin[i] : (K)0;
      v[r] = i < n ? vin[i] : 0u;
    }
#pragma unroll
    for (int r = 0; r < kMsItems; ++r) {
      const int i = tile0 + (warp * kMsItems + r) * 32 + lane;
      const bool valid = i < n;
      d[r] = valid ? (int)((k[r] >> shift) & 255) : 0;
      mk[r] = match_digit(d[r], valid);
      if (valid && lane == __ffs(mk[r]) - 1) warp_cnt[warp][d[r]] += __popc(mk[r]);
      __syncwarp();
    }
    __syncthreads();
    if (tid < 256) {
      // per digit: offsets of the warps inside the tile's run of that digit, then the runs' starts
      unsigned int run = 0;
#pragma unroll
      for (int q = 0; q < kMsWarps; ++q) {
        const unsigned int cnt = warp_cnt[q][tid];
        warp_cnt[q][tid] = run;
        run += cnt;
      }
      unsigned int x = run;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) wsum[warp] = x;
      tile_prefix[tid] = x - run;  // exclusive inside the warp; the warps before are added below
      gfirst[tid] = first_slot;
    }
    __syncthreads();
    if (tid < 256) {
      unsigned int add = 0;
      for (int q = 0; q < warp; ++q) add += wsum[q];
      tile_prefix[tid] += add;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kMsItems; ++r) {
      const int i = tile0 + (warp * kMsItems + r) * 32 + lane;
      const bool valid = i < n;
      const unsigned int mask = mk[r];
      const int leader = valid ? __ffs(mask) - 1 : lane;
      unsigned int pos = 0;
      if (valid && lane == leader) {
        pos = warp_cnt[warp][d[r]];
        warp_cnt[warp][d[r]] = pos + __popc(mask);
      }
      pos = __shfl_sync(0xffffffffu, pos, leader);
      if (valid) {
        const unsigned int lp = tile_prefix[d[r]] + pos + __popc(mask & ((1u << lane) - 1u));
        s_key[lp] = k[r];
        s_val[lp] = v[r];
      }
      __syncwarp();
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kMsItems; ++r) {
      const int j = r * kMsThreads + tid;
      if (j < tile_n) {
        const K kk = s_key[j];
        const int dd = (int)((kk >> shift) & 255);
        const unsigned int dst = gfirst[dd] + ((unsigned int)j - tile_prefix[dd]);
        kout[dst] = kk;
        vout[dst] = s_val[j];
      }
    }
    __syncthreads();
  }
}

template <typename K>
constexpr size_t ms_scatter_smem() {
  return (size_t)kMsTile * (sizeof(K) + 4) + (size_t)kMsWarps * 256 * 4 + 2 * 256 * 4 + 64;
}

// Host side.  `total` = upper bound of the elements in all segments (sizes the workspace),
// `ws` a buffer of the context that lives until the stream has run the sort.
template <typename K>
static inline int seg_sort_multi(const SegSortArgsT<K>& a, int nseg, int64_t total, int num_sms, cudaStream_t stream,
                                 DevBuf& ws, int64_t* launches) {
  if (nseg <= 0) return 0;
  const int npass = (a.hi_bit - a.lo_bit + 7) / 8;
  const int64_t max_tiles = total / kMsTile + nseg + 1;
  const size_t off_tseg = ((size_t)4 * (nseg + 1) + 255) & ~(size_t)255;
  const size_t off_counts = (off_tseg + (size_t)4 * max_tiles + 255) & ~(size_t)255;
  const size_t off_where = off_counts + (size_t)max_tiles * 1024;
  const size_t need = off_where + (size_t)3 * nseg + 256;
  if (ws.reserve(need)) return 1;
  char* p = ws.as<char>();
  MsWork w;
  w.tile_first = reinterpret_cast<int32_t*>(p);
  w.tile_seg = reinterpret_cast<int32_t*>(p + off_tseg);
  w.counts = reinterpret_cast<unsigned int*>(p + off_counts);
  unsigned char* wa = reinterpret_cast<unsigned char*>(p + off_where);
  unsigned char* wb = wa + nseg;
  w.skip = wb + nseg;
  w.nseg = nseg;
  cudaMemsetAsync(wa, 0, (size_t)nseg, stream);
  if (npass <= 0) {
    cudaMemsetAsync(a.where, 0, (size_t)nseg, stream);
    return 0;
  }
  k_ms_plan<<<1, 1024, 0, stream>>>(a.seg_cnt, nseg, w.tile_first);
  k_ms_tilemap<<<nseg, 256, 0, stream>>>(w);
  // persistent grids: as many CTAs as stay resident
  int per_sm_c = 1, per_sm_s = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_c, k_ms_count<K>, kMsThreads, 0);
  cudaFuncSetAttribute(k_ms_scatter<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ms_scatter_smem<K>());  // per device
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_s, k_ms_scatter<K>, kMsThreads, ms_scatter_smem<K>());
  const int64_t max_grid = std::max<int64_t>(1, max_tiles);
  const int grid_c = (int)std::min<int64_t>((int64_t)num_sms * std::max(per_sm_c, 1), max_grid);
  const int grid = (int)std::min<int64_t>((int64_t)num_sms * std::max(per_sm_s, 1), max_grid);
  if (launches) *launches += 3 * npass + 1;  // + the one the caller's scope counts
  for (int p2 = 0; p2 < npass; ++p2) {
    w.where_in = (p2 & 1) ? wb : wa;
    w.where_out = p2 == npass - 1 ? a.where : ((p2 & 1) ? wa : wb);
    const int shift = a.lo_bit + 8 * p2;
    k_ms_count<K><<<grid_c, kMsThreads, 0, stream>>>(a, w, shift);
    k_ms_scan<<<nseg, 256, 0, stream>>>(a.seg_cnt, w);
    k_ms_scatter<K><<<grid, kMsThreads, ms_scatter_smem<K>(), stream>>>(a, w, shift);
  }
  return 0;
}

// Picks the one-CTA-per-segment kernel or the multi-CTA passes.  total = upper bound of the
// elements over all segments.  Call inside a KLU_LAUNCH scope (the passes are timed as one entry).
template <typename K>
static inline int seg_sort_launch(klu_ctx* c, const SegSortArgsT<K>& a, int nseg, int64_t total) {
  if (nseg <= 0) return 0;
  static const bool single_only = getenv("KLU_SORT_SINGLE") != nullptr;
  static const bool multi_only = getenv("KLU_SORT_MULTI") != nullptr;  // tests
  // few segments of a few tiles at least, or very large ones; thousands of mid-sized segments (the
  // packer's sorts at 10 k lattices) run faster one CTA each (41 vs 54 ms)
  const int64_t avg = total / nseg;
  const bool multi = multi_only || (!single_only && avg >= 2 * kMsTile && (nseg < c->num_sms * 8 || avg >= 64 * kMsTile));
  if (!multi) {
    seg_sort_launch(a, nseg, c->stream);
    return 0;
  }
  return seg_sort_multi(a, nseg, total, c->num_sms, c->stream, c->d_sortws, &c->launches);
}

// After a sort that looked at the bits >= a.lo_bit only: every run of elements whose keys agree
// there is put in full-key order by a stable insertion sort, one thread per run (the runs are
// log-posteriors equal to ~1e-6 relative: a handful per segment).  Grid (segments, tiles);
// where[] as k_seg_radix_sort left it; seg0 = first segment of this launch.
static __global__ void __launch_bounds__(256) k_seg_order_fixup(SegSortArgs a, int seg0) {
  const int seg = seg0 + blockIdx.x;
  const int n = a.seg_cnt[seg];
  const int64_t base = a.seg_base[seg];
  unsigned long long* K = (a.where[seg] ? a.key_b : a.key_a) + base;
  unsigned int* V = (a.where[seg] ? a.val_b : a.val_a) + base;
  for (int i = blockIdx.y * blockDim.x + threadIdx.x; i + 1 < n; i += gridDim.y * blockDim.x) {
    const unsigned long long t = K[i] >> a.lo_bit;
    if ((i > 0 && (K[i - 1] >> a.lo_bit) == t) || (K[i + 1] >> a.lo_bit) != t) continue;  // not the head of a run
    int j = i + 1;
    while (j < n && (K[j] >> a.lo_bit) == t) {  // insert element j into the ordered [i, j)
      const unsigned long long k = K[j];
      const unsigned int v = V[j];
      int q = j;
      while (q > i && K[q - 1] > k) {
        K[q] = K[q - 1];
        V[q] = V[q - 1];
        --q;
      }
      K[q] = k;
      V[q] = v;
      ++j;
    }
  }
}
#endif

}  // namespace klu
