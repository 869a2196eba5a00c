// klu_lendist.cu -- lattice-to-transcript-length-dist (SURVEY.md 8f rank 4).
//
// Reference: latbin/lattice-to-transcript-length-dist.cc:64-125.  In the lattice that
// DisambiguateStateInputSequenceLength would unfold, every final state (len, u) adds
// fw[(len, u)] - cost(final(u)) to the length's accumulator; here that is the banded
// alpha of klu_sweep.cu read at the final states.  One warp per lattice, a lane per
// length; the final states are folded in input-state order (the unfolded lattice's id
// order for a fixed length).  Output = one Posterior frame per lattice:
// (length, float logp) sorted by (float logp desc, length asc).
#include <math.h>

#include <algorithm>

#include "klu_common.cuh"
#include "klu_sort.cuh"

namespace klu {

namespace {

struct LenArgs {
  BatchView b;
  CostParams cp;
  const double* alpha2;     // chunk-local banded alpha
  long long band_base;
  const double* total;
  const int64_t* ent_base;  // [L+1] slots per lattice: max_len + 1
  unsigned long long* key;
  unsigned int* val;
  int32_t* cnt;             // [L]
  int l0, l1;
};

__global__ void __launch_bounds__(128) k_len_emit(LenArgs a) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int l = a.l0 + warp;
  if (l >= a.l1) return;
  const BatchView& b = a.b;
  const int s0 = b.s_off[l], ns = b.s_off[l + 1] - s0;
  const int64_t base = a.ent_base[l];
  const int maxlen = (int)(a.ent_base[l + 1] - base) - 1;
  int n = 0;
  for (int len0 = 0; len0 <= maxlen; len0 += 32) {
    const int len = len0 + lane;
    double acc = neg_inf();
    if (len <= maxlen) {
      for (int si = 0; si < ns; ++si) {
        const int p = b.old2new[s0 + si];
        const float fg = b.fin_g[p], fa = b.fin_a[p];
        if (isinf(fg) && isinf(fa)) continue;
        const int lo = b.band_lo[p];
        const int w = (int)(b.band_off[p + 1] - b.band_off[p]);
        if (lo < 0 || len < lo || len >= lo + w) continue;
        const double x = a.alpha2[b.band_off[p] - a.band_base + (len - lo)];
        if (x > neg_inf()) acc = log_add(acc, x - final_cost(fg, fa, a.cp));
      }
    }
    const bool has = acc > neg_inf();
    const unsigned int bal = __ballot_sync(0xffffffffu, has);
    if (has) {
      const int slot = n + __popc(bal & ((1u << lane) - 1u));
      const float f = (float)(acc - a.total[l]) + 0.0f;
      a.key[base + slot] = ((unsigned long long)(~ord_f32(f)) << 32) | (unsigned int)len;
      a.val[base + slot] = (unsigned int)slot;
    }
    n += __popc(bal);
  }
  if (lane == 0) a.cnt[l] = n;
}

__global__ void __launch_bounds__(128) k_len_gather(const int64_t* ent_base, const int32_t* cnt, const int64_t* res_off,
                                                    const unsigned long long* key_a, const unsigned long long* key_b,
                                                    const unsigned char* where, int32_t* o_len, float* o_logp, int L) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= L) return;
  const unsigned long long* key = (where[warp] ? key_b : key_a) + ent_base[warp];
  const int64_t out = res_off[warp];
  for (int i = lane; i < cnt[warp]; i += 32) {
    const unsigned long long k = key[i];
    o_len[out + i] = (int32_t)(k & 0xffffffffu);
    const unsigned int u = ~(unsigned int)(k >> 32);
    o_logp[out + i] = __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
  }
}

}  // namespace

int run_length_dist(klu_ctx* c, const klu_opts* o) {
  const int32_t L = c->L;
  CostParams cp = make_cost_params(o, false);
  KLU_TRY(run_log_sweeps(c, cp, false, 0.f));
  c->h_res_off.assign(L + 1, 0);
  c->last_entries = 0;
  if (L == 0) return 0;
  std::vector<int64_t> ent_base(L + 1, 0);
  for (int32_t l = 0; l < L; ++l) ent_base[l + 1] = ent_base[l] + c->h_maxlen[l] + 1;
  const size_t N = (size_t)ent_base[L];
  enum { S_BASE = 0, S_KEYA, S_KEYB, S_VALA, S_VALB, S_CNT, S_WHERE };
  DevBuf* sc = c->d_scratch;
  KLU_TRY(sc[S_BASE].reserve(8 * (size_t)(L + 1)));
  KLU_TRY(sc[S_KEYA].reserve(8 * N));
  KLU_TRY(sc[S_KEYB].reserve(8 * N));
  KLU_TRY(sc[S_VALA].reserve(4 * N));
  KLU_TRY(sc[S_VALB].reserve(4 * N));
  KLU_TRY(sc[S_CNT].reserve(4 * (size_t)L));
  KLU_TRY(sc[S_WHERE].reserve((size_t)L));
  KLU_TRY(c->d_res[5].reserve(8 * (size_t)(L + 1)));
  KLU_TRY(c->d_res[0].reserve(4 * N));
  KLU_TRY(c->d_res[4].reserve(4 * N));
  KLU_CUDA(cudaMemcpyAsync(sc[S_BASE].p, ent_base.data(), 8 * (size_t)(L + 1), cudaMemcpyHostToDevice, c->stream));
  KLU_CUDA(cudaStreamSynchronize(c->stream));
  LenArgs a;
  a.b = c->view();
  a.cp = cp;
  a.total = c->d_total.as<double>();
  a.ent_base = sc[S_BASE].as<int64_t>();
  a.key = sc[S_KEYA].as<unsigned long long>();
  a.val = sc[S_VALA].as<unsigned int>();
  a.cnt = sc[S_CNT].as<int32_t>();
  // chunks of lattices whose (state, length) bands fit the banded-alpha buffer
  const int64_t kBandBudget = (int64_t)1 << 30;
  for (int32_t l0 = 0; l0 < L;) {
    int32_t l1 = l0 + 1;
    while (l1 < L && c->h_band_off[l1 + 1] - c->h_band_off[l0] <= kBandBudget) ++l1;
    KLU_TRY(run_banded_alpha(c, cp, false, 0.f, l0, l1));
    a.alpha2 = c->d_alpha2.as<double>();
    a.band_base = c->h_band_off[l0];
    a.l0 = l0;
    a.l1 = l1;
    {
      KLU_LAUNCH(c, "k_len_emit");
      k_len_emit<<<((l1 - l0) * 32 + 127) / 128, 128, 0, c->stream>>>(a);
    }
    KLU_TRY(check_launch("k_len_emit"));
    l0 = l1;
  }
  SegSortArgs ss;
  ss.seg_base = a.ent_base;
  ss.seg_cnt = a.cnt;
  ss.key_a = sc[S_KEYA].as<unsigned long long>();
  ss.val_a = sc[S_VALA].as<unsigned int>();
  ss.key_b = sc[S_KEYB].as<unsigned long long>();
  ss.val_b = sc[S_VALB].as<unsigned int>();
  ss.where = sc[S_WHERE].as<unsigned char>();
  ss.lo_bit = 0;
  ss.hi_bit = 64;
  {
    KLU_LAUNCH(c, "k_seg_radix_sort");
    seg_sort_launch(ss, L, c->stream);
  }
  KLU_TRY(check_launch("k_seg_radix_sort(length dist)"));
  KLU_TRY(scan_counts(c, a.cnt, 0, L, c->d_res[5].as<int64_t>(), "k_len_scan"));
  {
    KLU_LAUNCH(c, "k_len_gather");
    k_len_gather<<<(L * 32 + 127) / 128, 128, 0, c->stream>>>(a.ent_base, a.cnt, c->d_res[5].as<int64_t>(), ss.key_a, ss.key_b,
                                                              ss.where, c->d_res[0].as<int32_t>(), c->d_res[4].as<float>(), L);
  }
  KLU_TRY(check_launch("k_len_gather"));
  c->last_entries = -1;  // offsets are read back lazily (klu_result_offsets)
  return 0;
}

}  // namespace klu
