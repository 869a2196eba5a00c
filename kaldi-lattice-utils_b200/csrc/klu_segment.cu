// klu_segment.cu -- lattice-word-index-segment without a global sort by key.
//
//   kwsbin2/lattice-word-index-segment.cc:134-177 (accumulate into a std::map keyed by
//   (word, t0, t1)), :96-128 (flatten, sort by logp desc, word, t0, t1)
//
// Two arcs can only share a key when they START AT THE SAME FRAME.  So instead of sorting
// all the arcs of a lattice by their 64-bit key (five radix passes in the generic pipeline of
// klu_index.cu), the arcs are bucketed by start frame once per batch (a stable 32-bit radix
// sort of E frame numbers + bucket offsets: structure only, klu_load_times reports it with the
// other per-batch indexes) and every run sorts each bucket -- the ~80 arcs that start in one
// frame -- by (word, duration) in shared memory: one warp per bucket, a bitonic network over
// 64-bit words {key, arc rank}, then the run heads fold their arcs with LogAdd in arc order.
// The reduced entries land in an arena indexed like the sorted arcs (a bucket's entries at the
// start of its arc range), a per-lattice scan of the buckets' entry counts packs their (order key,
// arena index) pairs back to back, and the order sort by log-posterior runs on those.
//
// Buckets larger than kBucketCap arcs (or keys that do not fit) send the whole batch through
// the generic pipeline instead (run_index_tool) -- e.g. a lattice with hundreds of parallel arcs
// between two states.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

constexpr int kBucketCap = 512;   // arcs of one lattice starting in one frame
constexpr int kBucketWarps = 8;   // per CTA; 16 B of shared memory per warp and bucket slot

struct SegArgs {
  BatchView b;
  CostParams cp;
  int filter_mode, filter_n;
  const int32_t* filter;
  const double* alpha;
  const double* beta;
  const double* total;
  int use_beam;
  const double* vfwd;
  const double* vbwd;
  const double* best;
  double beam;
  int bits_label, bits_time, bits_span;
  // per batch
  const int32_t* slot_base;  // [L+1] first bucket slot of each lattice (max time + 2 slots each)
  const int32_t* boff;       // per slot: first sorted arc (global arc index) of the bucket
  const unsigned int* perm_a;  // sorted arcs -> out-order arc (lattice-local), in whichever buffer the sort left them
  const unsigned int* perm_b;
  const unsigned char* where;
  int num_slots;
  // per run: the arena (indexed like the sorted arcs)
  ulonglong2* rec;       // {key (word, t0, span), bits of the log-posterior}
  int tiles;             // CTAs per lattice
  int cap;               // shared-memory slots per warp: power of two >= the largest bucket
  int rank_bits;         // log2(cap): low bits of a sort word = the arc's rank in its bucket
  unsigned int* key32;   // order keys (high half of the f64 key), at arena positions
  unsigned int* idx;     // lattice-local arena index
  int32_t* rcnt;         // [L] entries
  int32_t* slot_cnt;     // per bucket slot: entries (run heads) it produced
  int32_t* slot_dense;   // per bucket slot: lattice-local first dense position of its entries
  unsigned int* key32_d;  // dense copies of key32 / idx (what the order sort works on)
  unsigned int* idx_d;
};

__device__ __forceinline__ bool seg_label_valid(const SegArgs& a, int label) {
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

// grid (lattices, tiles): sort keys of the bucketing = start frame of every out-order arc
// (flags[1] is raised by an arc between states without a time -- unreachable ones: the generic
// pipeline keeps the reference's behaviour for those)
__global__ void __launch_bounds__(256) k_sg_time_keys(BatchView b, unsigned int* key, unsigned int* val, int* flags) {
  const int l = blockIdx.x;
  const int e0 = b.e_off[l], e1 = b.e_off[l + 1];
  for (int e = e0 + blockIdx.y * blockDim.x + threadIdx.x; e < e1; e += gridDim.y * blockDim.x) {
    const int t0 = b.time[b.out_src[e]], t1 = b.time[b.out_rec[e].x];
    if (t0 < 0 || t1 < t0) flags[1] = 1;
    key[e] = (unsigned int)max(t0, 0);
    val[e] = (unsigned int)(e - e0);
  }
}

// one thread per bucket slot: first sorted arc whose start frame is >= the slot's frame
__global__ void __launch_bounds__(256) k_sg_bucket_offsets(BatchView b, const int32_t* slot_base, const unsigned int* key_a,
                                                           const unsigned int* key_b, const unsigned char* where,
                                                           int num_slots, int32_t* boff, int* max_bucket) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  int mine = 0;
  if (slot < num_slots) {
    const int l = last_le(slot_base, 0, b.L - 1, slot);  // lattice of the slot
    const unsigned int k = (unsigned int)(slot - slot_base[l]);
    const int e0 = b.e_off[l], n = b.e_off[l + 1] - e0;
    const unsigned int* key = (where[l] ? key_b : key_a) + e0;
    auto lower = [&](unsigned int x) {
      int a0 = 0, a1 = n;  // first j with key[j] >= x
      while (a0 < a1) {
        const int mid = (a0 + a1) >> 1;
        if (key[mid] < x) a0 = mid + 1;
        else a1 = mid;
      }
      return a0;
    };
    const int first = lower(k);
    boff[slot] = e0 + first;
    mine = lower(k + 1) - first;
    if (slot == num_slots - 1) boff[num_slots] = b.E;
  }
  mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, 16));
  mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, 8));
  mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, 4));
  mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, 2));
  mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, 1));
  if ((threadIdx.x & 31) == 0 && mine > 0) atomicMax(max_bucket, mine);
}

// Streaming log-sum-exp over the values of one key run (see klu_index.cu RunSum)
struct SegRunSum {
  double m, s;
  __device__ SegRunSum() : m(neg_inf()), s(0.0) {}
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

// One warp per bucket (the arcs of a lattice that start in one frame).  Grid lattices x tiles, tile fastest:
// the CTAs running at the same time work on a few lattices, whose alpha / beta / times stay in L2.
// KT: 32-bit sort words when (word, span, rank) fit (half the shared-memory traffic of the network)
template <typename KT>
__global__ void __launch_bounds__(kBucketWarps * 32) k_sg_buckets(SegArgs a) {
  extern __shared__ unsigned long long s_dyn[];
  constexpr KT kNoKey = (KT)~(KT)0;
  const int kRankBits = a.rank_bits;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* sv = reinterpret_cast<double*>(s_dyn) + (size_t)warp * a.cap;
  KT* sk = reinterpret_cast<KT*>(s_dyn + (size_t)kBucketWarps * a.cap) + (size_t)warp * a.cap;
  const BatchView& b = a.b;
  const int l = blockIdx.x / a.tiles, tile = blockIdx.x % a.tiles;  // tile fastest: see above
  const int e0 = b.e_off[l];
  const int slot0 = a.slot_base[l], nslots = a.slot_base[l + 1] - slot0;
  const unsigned int* perm = (a.where[l] ? a.perm_b : a.perm_a);
  const double total = a.total[l];
  for (int f = tile * kBucketWarps + warp; f < nslots; f += a.tiles * kBucketWarps) {
    const int slot = slot0 + f;
    const int j0 = a.boff[slot], n = a.boff[slot + 1] - j0;
    if (n <= 0) {
      if (lane == 0) a.slot_cnt[slot] = 0;
      continue;
    }
    const unsigned long long t0 = (unsigned long long)f;
    int P = 32;
    while (P < n) P <<= 1;
    // ---- keys {(word, span), arc rank in the bucket} and values of the bucket's arcs
    for (int j = lane; j < P; j += 32) {
      KT k = kNoKey;
      double v = neg_inf();
      if (j < n) {
        const int e = e0 + (int)perm[j0 + j];
        const int4 r = b.out_rec[e];
        const int s = b.out_src[e];
        bool valid = seg_label_valid(a, r.w);
        if (valid && a.use_beam) {  // PruneLattice [ext] drops the arc
          CostParams cp = a.cp;
          cp.float_sum = 0;
          const double fb = __dadd_rn(a.vfwd[s], __dadd_rn(rec_cost(r, cp), a.vbwd[r.x]));
          if (fb > __dadd_rn(a.best[l], a.beam)) valid = false;
        }
        if (valid) {
          // fw[s] + arc_lkh + bw[next], kwsbin2/lattice-word-index-segment.cc:160-162
          v = __dadd_rn(__dadd_rn(a.alpha[s], -rec_cost(r, a.cp)), a.beta[r.x]);
          const unsigned long long span = (unsigned long long)(b.time[r.x] - b.time[s]);
          k = (KT)((((((unsigned long long)(unsigned int)r.w) << a.bits_span) | span) << kRankBits) | (unsigned long long)j);
        }
      }
      sk[j] = k;
      sv[j] = v;
    }
    __syncwarp();
    // ---- bitonic sort of the P keys (ascending); the low bits keep equal (word, span) in arc order
    for (int size = 2; size <= P; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        for (int t = lane; t < (P >> 1); t += 32) {
          const int i = (t << 1) - (t & (stride - 1));  // stride is a power of two
          const int p = i + stride;
          const bool up = ((i & size) == 0);
          const KT x = sk[i], y = sk[p];
          if ((x > y) == up) {
            sk[i] = y;
            sk[p] = x;
          }
        }
        __syncwarp();
      }
    }
    // ---- run heads fold their arcs (LogAdd in arc order), entries to the arena
    int carry = 0;
    for (int i0 = 0; i0 < P; i0 += 32) {
      const int i = i0 + lane;
      const KT k = sk[i];
      const bool head = k != kNoKey && (i == 0 || (sk[i - 1] >> kRankBits) != (k >> kRankBits));
      const unsigned int hm = __ballot_sync(0xffffffffu, head);
      if (head) {
        const int rank = carry + __popc(hm & ((1u << lane) - 1u));
        double sum = sv[(int)(k & (KT)(a.cap - 1))];
        int q = i + 1;
        if (q + 1 < P && (sk[q + 1] >> kRankBits) == (k >> kRankBits)) {  // three or more terms
          SegRunSum rs;
          rs.add(sum);
          for (; q < P && (sk[q] >> kRankBits) == (k >> kRankBits); ++q) rs.add(sv[(int)(sk[q] & (KT)(a.cap - 1))]);
          sum = rs.value();
        } else {
          for (; q < P && (sk[q] >> kRankBits) == (k >> kRankBits); ++q) sum = log_add(sum, sv[(int)(sk[q] & (KT)(a.cap - 1))]);
        }
        const double logp = sum - total;
        const unsigned long long ws = (unsigned long long)(k >> kRankBits);  // (word, span)
        const unsigned long long word = ws >> a.bits_span, span = ws & ((1ULL << a.bits_span) - 1ULL);
        a.rec[j0 + rank] = make_ulonglong2((((word << a.bits_time) | t0) << a.bits_span) | span,
                                           (unsigned long long)__double_as_longlong(logp));
        a.key32[j0 + rank] = (unsigned int)((~ord_f64(logp + 0.0)) >> 32);
        a.idx[j0 + rank] = (unsigned int)(j0 + rank - e0);
      }
      carry += __popc(hm);
    }
    if (lane == 0) a.slot_cnt[slot] = carry;  // the rest of the bucket's arena range stays unused
    __syncwarp();
  }
}

// one CTA per lattice: exclusive scan of its buckets' entry counts -> where each bucket's entries go
// in the dense order-sort input; the lattice's entry count
__global__ void __launch_bounds__(256) k_sg_dense_offsets(SegArgs a) {
  __shared__ int warp_sum[8];
  __shared__ int carry_s;
  const int l = blockIdx.x;
  const int slot0 = a.slot_base[l], nslots = a.slot_base[l + 1] - slot0;
  const int tid = threadIdx.x;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < nslots; base += 256) {
    const int i = base + tid;
    const int c = i < nslots ? a.slot_cnt[slot0 + i] : 0;
    const int pre = cta_exclusive_scan<int, 256>(c, warp_sum, carry_s);
    if (i < nslots) a.slot_dense[slot0 + i] = pre;
  }
  if (tid == 0) a.rcnt[l] = carry_s;
}

// one warp per bucket: its entries' (order key, arena index) pairs to the dense arrays
template <typename KT>
__global__ void __launch_bounds__(kBucketWarps * 32) k_sg_densify(SegArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int l = blockIdx.x / a.tiles, tile = blockIdx.x % a.tiles;
  const int e0 = a.b.e_off[l];
  const int slot0 = a.slot_base[l], nslots = a.slot_base[l + 1] - slot0;
  for (int f = tile * kBucketWarps + warp; f < nslots; f += a.tiles * kBucketWarps) {
    const int slot = slot0 + f;
    const int cnt = a.slot_cnt[slot];
    const int j0 = a.boff[slot], d0 = e0 + a.slot_dense[slot];
    for (int r = lane; r < cnt; r += 32) {
      a.key32_d[d0 + r] = a.key32[j0 + r];
      a.idx_d[d0 + r] = a.idx[j0 + r];
    }
  }
}

// After the 32-bit order sort: runs of equal high halves are put in the reference's full
// order -- (logp desc, word, t0, t1) -- by a stable insertion sort, one thread per run.
struct SegFixArgs {
  const int64_t* seg_base;
  const int32_t* seg_cnt;
  const unsigned char* where;
  const unsigned int *key_a, *key_b;
  unsigned int *val_a, *val_b;
  const ulonglong2* rec;
  int tiles;
};

__global__ void __launch_bounds__(256) k_sg_order_fixup(SegFixArgs a) {
  const int l = blockIdx.x / a.tiles, tile = blockIdx.x % a.tiles;
  const int n = a.seg_cnt[l];
  const int64_t base = a.seg_base[l];
  const unsigned int* K = (a.where[l] ? a.key_b : a.key_a) + base;
  unsigned int* V = (a.where[l] ? a.val_b : a.val_a) + base;
  const ulonglong2* rec = a.rec + base;
  for (int i = tile * blockDim.x + threadIdx.x; i + 1 < n; i += a.tiles * blockDim.x) {
    const unsigned int t = K[i];
    if (t == 0xffffffffu) continue;
    if ((i > 0 && K[i - 1] == t) || K[i + 1] != t) continue;  // not the head of a run
    int j = i + 1;
    while (j < n && K[j] == t) {  // insert element j into the ordered [i, j)
      const unsigned int v = V[j];
      const ulonglong2 rv = rec[v];
      const unsigned long long k = ~ord_f64(__longlong_as_double((long long)rv.y) + 0.0), kk = rv.x;
      int q = j;
      while (q > i) {
        const unsigned int u = V[q - 1];
        const ulonglong2 ru = rec[u];
        const unsigned long long ku = ~ord_f64(__longlong_as_double((long long)ru.y) + 0.0);
        if (ku < k || (ku == k && ru.x <= kk)) break;
        V[q] = u;
        --q;
      }
      V[q] = v;
      ++j;
    }
  }
}

struct SegGatherArgs {
  BatchView b;
  const int64_t* seg_base;
  const int32_t* rcnt;
  const int64_t* res_off;
  const unsigned char* where;
  const unsigned int *idx_a, *idx_b;
  const ulonglong2* rec;
  int bits_time, bits_span, tiles;
  int32_t *c0, *c1, *c2;
  double* v;
};

__global__ void __launch_bounds__(256) k_sg_gather(SegGatherArgs a) {
  const int l = blockIdx.x / a.tiles, tile = blockIdx.x % a.tiles;
  const int n = a.rcnt[l];
  const int64_t base = a.seg_base[l];
  const int64_t out = a.res_off[l];
  const unsigned int* idx = (a.where[l] ? a.idx_b : a.idx_a) + base;
  const unsigned long long tm = (1ULL << a.bits_time) - 1ULL, sm = (1ULL << a.bits_span) - 1ULL;
  for (int i = tile * blockDim.x + threadIdx.x; i < n; i += a.tiles * blockDim.x) {
    const ulonglong2 r = a.rec[base + idx[i]];
    const unsigned long long k = r.x;
    const int32_t t0 = (int32_t)((k >> a.bits_span) & tm);
    a.c0[out + i] = (int32_t)(k >> (a.bits_time + a.bits_span));
    a.c1[out + i] = t0;
    a.c2[out + i] = t0 + (int32_t)(k & sm);
    a.v[out + i] = __longlong_as_double((long long)r.y);
  }
}

int bits_for(int64_t maxv) {
  int b = 1;
  while (b < 63 && ((int64_t)1 << b) <= maxv) ++b;
  return b;
}

}  // namespace

// The arcs of the loaded batch bucketed by start frame (structure only: built on first use).
// Sets c->seg_max_bucket; the caller falls back to the generic pipeline when it exceeds the cap.
int ensure_segment_buckets(klu_ctx* c) {
  if (c->seg_ready) return 0;
  const int32_t L = c->L;
  KLU_CUDA(cudaEventRecord(c->ev_p0, c->stream));
  const size_t E1 = (size_t)std::max<int64_t>(c->E, 1);
  std::vector<int32_t> slot_base(L + 1, 0), seg_cnt(L);
  int64_t slots = 0, max_arcs = 0;
  for (int32_t l = 0; l < L; ++l) {
    slot_base[l] = (int32_t)slots;
    slots += (int64_t)c->h_maxtime[l] + 2;
    seg_cnt[l] = (int32_t)(c->h_e_off[l + 1] - c->h_e_off[l]);
    max_arcs = std::max<int64_t>(max_arcs, seg_cnt[l]);
  }
  slot_base[L] = (int32_t)slots;
  if (slots >= ((int64_t)1 << 31) - 2) {
    c->seg_max_bucket = 0x7fffffff;  // generic pipeline
    c->seg_ready = true;
    return 0;
  }
  c->seg_slots = (int32_t)slots;
  // key / permutation ping-pong buffers live in the tool scratch (free between runs); what stays:
  // the permutation (4 B/arc, in whichever buffer the sort left it -> copied to d_sg_perm), bucket offsets
  DevBuf* sc = c->d_scratch;
  KLU_TRY(sc[0].reserve(4 * E1));
  KLU_TRY(sc[1].reserve(4 * E1));
  KLU_TRY(c->d_sg_meta.reserve(4 * (size_t)(L + 1) + 8 * (size_t)(L + 1) + 4 * (size_t)L + 2 * (size_t)L + 64));
  int32_t* d_slot_base = c->d_sg_meta.as<int32_t>();
  int64_t* d_seg_base = reinterpret_cast<int64_t*>(d_slot_base + (L + 1) + ((L + 1) & 1));
  int32_t* d_seg_cnt = reinterpret_cast<int32_t*>(d_seg_base + L + 1);
  unsigned char* d_where = reinterpret_cast<unsigned char*>(d_seg_cnt + L);
  KLU_TRY(c->d_sg_boff.reserve(4 * (size_t)(slots + 2)));
  KLU_TRY(c->d_sg_perm.reserve(2 * 4 * E1));  // both sort buffers of the permutation side
  KLU_TRY(c->d_counter.reserve(64));
  KLU_CUDA(cudaMemsetAsync(c->d_counter.p, 0, 64, c->stream));
  KLU_CUDA(cudaMemcpyAsync(d_slot_base, slot_base.data(), 4 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemcpyAsync(d_seg_base, c->h_e_off.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaMemcpyAsync(d_seg_cnt, seg_cnt.data(), 4 * (size_t)L, cudaMemcpyHostToDevice, c->stream));
  const BatchView b = c->view();
  unsigned int* key_a = sc[0].as<unsigned int>();
  unsigned int* key_b = sc[1].as<unsigned int>();
  unsigned int* perm_a = c->d_sg_perm.as<unsigned int>();
  unsigned int* perm_b = perm_a + E1;
  const int tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  if (L > 0 && c->E > 0) {
    {
      KLU_LAUNCH(c, "k_sg_time_keys");
      k_sg_time_keys<<<dim3(L, tiles), 256, 0, c->stream>>>(b, key_a, perm_a, c->d_counter.as<int>());
    }
    KLU_TRY(check_launch("k_sg_time_keys"));
    SegSortArgs32 ss;
    ss.seg_base = d_seg_base;
    ss.seg_cnt = d_seg_cnt;
    ss.key_a = key_a;
    ss.val_a = perm_a;
    ss.key_b = key_b;
    ss.val_b = perm_b;
    ss.where = d_where;
    ss.lo_bit = 0;
    ss.hi_bit = std::min(32, bits_for(c->max_time));
    {
      KLU_LAUNCH(c, "k_seg_radix_sort");
      KLU_TRY(seg_sort_launch(c, ss, L, c->E));
    }
    KLU_TRY(check_launch("k_seg_radix_sort(start frames)"));
    {
      KLU_LAUNCH(c, "k_sg_bucket_offsets");
      k_sg_bucket_offsets<<<(int)((slots + 255) / 256), 256, 0, c->stream>>>(b, d_slot_base, key_a, key_b, d_where, (int)slots,
                                                                            c->d_sg_boff.as<int32_t>(), c->d_counter.as<int>());
    }
    KLU_TRY(check_launch("k_sg_bucket_offsets"));
  }
  int flags[2] = {0, 0};  // largest bucket, arcs without usable times
  KLU_CUDA(cudaMemcpyAsync(flags, c->d_counter.p, 8, cudaMemcpyDeviceToHost, c->stream));
  KLU_CUDA(cudaEventRecord(c->ev_p1, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->ev_p0, c->ev_p1);
  c->lazy_pack_ms += ms;
  c->seg_max_bucket = flags[1] ? 0x7fffffff : flags[0];
  c->seg_ready = true;
  {
    char msg[96];
    snprintf(msg, sizeof(msg), "segment buckets: %d slots, largest %d arcs, %.2f ms", (int)slots, c->seg_max_bucket, ms);
    klu_trace(c, msg);
  }
  return 0;
}

// Returns 1 when the fast path does not apply (the caller runs the generic pipeline), 0 when the
// results are in place, < 0 ... errors are reported through the usual non-zero return of KLU_TRY.
int run_segment_buckets(klu_ctx* c, const klu_opts* o, bool* done) {
  *done = false;
  const int32_t L = c->L;
  if (L == 0 || c->E == 0 || getenv("KLU_GENERIC_SEGMENT")) return 0;
  for (int32_t l = 0; l < L; ++l)
    if (!c->h_times_ok[l]) return 0;  // the generic path reports the error
  const int bits_label = bits_for(c->max_label), bits_time = bits_for(c->max_time), bits_span = bits_for(c->max_span);
  if (bits_label + bits_span + 9 > 63 || bits_label + bits_time + bits_span > 62) return 0;  // 9 = log2(kBucketCap)
  KLU_TRY(ensure_segment_buckets(c));
  if (c->seg_max_bucket > kBucketCap) return 0;
  const bool use_beam = o->beam != INFINITY;
  if (use_beam && !(o->beam > 0.0f)) {
    set_error("--beam must be positive");  // KALDI_ASSERT(beam > 0.0) in PruneLattice [ext]
    return 1;
  }
  const CostParams cp = make_cost_params(o, false);
  if (use_beam) KLU_TRY(run_tropical_sweeps(c, cp));
  KLU_TRY(run_log_sweeps(c, cp, use_beam, o->beam));
  const size_t E1 = (size_t)c->E;
  DevBuf* sc = c->d_scratch;
  enum { S_REC = 4, S_K32A, S_K32B, S_IDXA, S_IDXB, S_RCNT, S_SLOTS };
  KLU_TRY(sc[S_REC].reserve(16 * E1));
  KLU_TRY(sc[S_K32A].reserve(4 * E1));
  KLU_TRY(sc[S_K32B].reserve(4 * E1));
  KLU_TRY(sc[S_IDXA].reserve(4 * E1));
  KLU_TRY(sc[S_IDXB].reserve(4 * E1));
  KLU_TRY(sc[S_RCNT].reserve(4 * (size_t)L + (size_t)L + 64));
  KLU_TRY(sc[S_SLOTS].reserve(8 * ((size_t)c->seg_slots + 2)));
  KLU_TRY(c->d_res[5].reserve(8 * (size_t)(L + 1)));
  int fmode = 0, fn = 0;
  KLU_TRY(upload_filter(c, o, &fmode, &fn));
  int32_t* d_slot_base = c->d_sg_meta.as<int32_t>();
  int64_t* d_seg_base = reinterpret_cast<int64_t*>(d_slot_base + (L + 1) + ((L + 1) & 1));
  int32_t* d_seg_cnt = reinterpret_cast<int32_t*>(d_seg_base + L + 1);
  unsigned char* d_where = reinterpret_cast<unsigned char*>(d_seg_cnt + L);
  SegArgs a;
  memset(&a, 0, sizeof(a));
  a.b = c->view();
  a.cp = cp;
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
  a.bits_label = bits_label;
  a.bits_time = bits_time;
  a.bits_span = bits_span;
  a.slot_base = d_slot_base;
  a.boff = c->d_sg_boff.as<int32_t>();
  a.perm_a = c->d_sg_perm.as<unsigned int>();
  a.perm_b = a.perm_a + E1;
  a.where = d_where;
  a.num_slots = c->seg_slots;
  a.rec = sc[S_REC].as<ulonglong2>();
  a.cap = 32;
  a.rank_bits = 5;
  while (a.cap < c->seg_max_bucket) {
    a.cap <<= 1;
    ++a.rank_bits;
  }
  const bool narrow = bits_label + bits_span + a.rank_bits <= 31;
  a.key32 = sc[S_K32A].as<unsigned int>();
  a.idx = sc[S_IDXA].as<unsigned int>();
  a.rcnt = sc[S_RCNT].as<int32_t>();
  a.slot_cnt = sc[S_SLOTS].as<int32_t>();
  a.slot_dense = a.slot_cnt + c->seg_slots + 1;
  a.key32_d = sc[S_K32B].as<unsigned int>();
  a.idx_d = sc[S_IDXB].as<unsigned int>();
  unsigned char* where2 = reinterpret_cast<unsigned char*>(a.rcnt + L);
  {
    KLU_LAUNCH(c, "k_sg_buckets");
    int max_slots = 1;
    for (int32_t l = 0; l < L; ++l) max_slots = std::max(max_slots, c->h_maxtime[l] + 2);
    const int btiles = std::max(1, std::min((max_slots + kBucketWarps * 4 - 1) / (kBucketWarps * 4), 64));
    a.tiles = btiles;
    if (narrow) {
      KLU_CUDA(cudaFuncSetAttribute(k_sg_buckets<unsigned int>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kBucketWarps * kBucketCap * 12));  // per device
      k_sg_buckets<unsigned int><<<(unsigned int)((int64_t)L * btiles), kBucketWarps * 32, (size_t)kBucketWarps * a.cap * 12, c->stream>>>(a);
    } else {
      KLU_CUDA(cudaFuncSetAttribute(k_sg_buckets<unsigned long long>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kBucketWarps * kBucketCap * 16));
      k_sg_buckets<unsigned long long><<<(unsigned int)((int64_t)L * btiles), kBucketWarps * 32, (size_t)kBucketWarps * a.cap * 16, c->stream>>>(a);
    }
  }
  KLU_TRY(check_launch("k_sg_buckets"));
  // the entries (~0.7 per arc) back to back per lattice: the order sort moves no holes
  {
    KLU_LAUNCH(c, "k_sg_dense_offsets");
    k_sg_dense_offsets<<<L, 256, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_sg_dense_offsets"));
  {
    KLU_LAUNCH(c, "k_sg_densify");
    k_sg_densify<unsigned int><<<(unsigned int)((int64_t)L * a.tiles), kBucketWarps * 32, 0, c->stream>>>(a);
  }
  KLU_TRY(check_launch("k_sg_densify"));
  SegSortArgs32 s2;
  s2.seg_base = d_seg_base;
  s2.seg_cnt = a.rcnt;
  s2.key_a = a.key32_d;
  s2.val_a = a.idx_d;
  s2.key_b = a.key32;
  s2.val_b = a.idx;
  s2.where = where2;
  s2.lo_bit = 0;
  s2.hi_bit = 32;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    KLU_TRY(seg_sort_launch(c, s2, L, c->E));
  }
  KLU_TRY(check_launch("k_seg_radix_sort(order)"));
  int64_t max_arcs = 0;
  for (int32_t l = 0; l < L; ++l) max_arcs = std::max(max_arcs, c->h_e_off[l + 1] - c->h_e_off[l]);
  const int tiles = (int)std::max<int64_t>(1, std::min<int64_t>((max_arcs + 255) / 256, 64));
  SegFixArgs f;
  f.seg_base = d_seg_base;
  f.seg_cnt = a.rcnt;
  f.where = where2;
  f.key_a = s2.key_a;
  f.key_b = s2.key_b;
  f.val_a = s2.val_a;
  f.val_b = s2.val_b;
  f.rec = a.rec;
  f.tiles = tiles;
  {
    KLU_LAUNCH(c, "k_order_fixup");
    k_sg_order_fixup<<<(unsigned int)((int64_t)L * tiles), 256, 0, c->stream>>>(f);
  }
  KLU_TRY(check_launch("k_order_fixup"));
  KLU_TRY(scan_counts(c, a.rcnt, 0, L, c->d_res[5].as<int64_t>(), "k_scan_counts"));
  // result columns: at most one entry per arc
  KLU_TRY(c->d_res[0].reserve(4 * E1));
  KLU_TRY(c->d_res[1].reserve(4 * E1));
  KLU_TRY(c->d_res[2].reserve(4 * E1));
  KLU_TRY(c->d_res[4].reserve(8 * E1));
  SegGatherArgs g;
  g.b = a.b;
  g.seg_base = d_seg_base;
  g.rcnt = a.rcnt;
  g.res_off = c->d_res[5].as<int64_t>();
  g.where = where2;
  g.idx_a = s2.val_a;
  g.idx_b = s2.val_b;
  g.rec = a.rec;
  g.tiles = tiles;
  g.bits_time = bits_time;
  g.bits_span = bits_span;
  g.c0 = c->d_res[0].as<int32_t>();
  g.c1 = c->d_res[1].as<int32_t>();
  g.c2 = c->d_res[2].as<int32_t>();
  g.v = c->d_res[4].as<double>();
  {
    KLU_LAUNCH(c, "k_gather");
    k_sg_gather<<<(unsigned int)((int64_t)L * tiles), 256, 0, c->stream>>>(g);
  }
  KLU_TRY(check_launch("k_gather"));
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = -1;  // known after klu_result_offsets()
  *done = true;
  return 0;
}

}  // namespace klu
