// klu_pack.cu -- lattice packer (north_star subsystem 1, SURVEY.md K0).
//
// Replaces what the reference does implicitly with VectorFst copies
// (kwsbin2/lattice-word-index-position.cc:64,93; TopSortCompactLatticeIfNeeded
// [ext]; CompactLatticeStateTimes [ext] kwsbin2/lattice-word-index-position.cc:67):
// a batch of CompactLattices becomes
//   * states renumbered per lattice by (level, input id), level = longest arc
//     distance from a source state  -> every level is a contiguous state range
//     whose incoming arcs all start in earlier levels (the "frontier offsets");
//   * arcs twice, as 16-byte records {peer state, graph, acoustic, label}:
//     sorted by destination (pull order of the forward sweep) and by source
//     (pull order of the backward sweep, emit order of the index kernels);
//   * per state: CSR offsets, final weights, frame time, input id, and the band
//     [lo, hi] of possible #non-epsilon labels on paths from the start (the
//     length axis of fstext/fstext-utils2.h:109-215, never materialised).
// Host threads pack disjoint lattice ranges; one cudaMemcpyAsync per array.
#include <string.h>

#include <cmath>

#include <algorithm>
#include <numeric>
#include <thread>

#include "klu_common.cuh"

namespace klu {

namespace {

struct Staging {
  std::vector<int32_t> s_off, e_off, lvl_off, lvl_start, in_off, out_off, out_src, out_orig, in2out, time, orig, level, band_lo,
      order;
  std::vector<int64_t> band_off;
  std::vector<int4> in_rec, out_rec;
  std::vector<float> fin_g, fin_a;
};

struct LatInfo {
  int32_t nl = 0;
  int32_t num_frames = 0;
  uint8_t times_ok = 1;
  int32_t max_label = 0, max_time = 0, max_len = 0, max_indeg = 0, max_outdeg = 0, max_span = 0;
  int64_t cap_frame = 0, cap_pos = 0, band = 0;
  std::string err;
};

inline int32_t f2i(float f) {
  int32_t i;
  memcpy(&i, &f, 4);
  return i;
}

// Pass 1 (per lattice): validate, levels.  Returns number of levels.
void lattice_levels(const klu_lattices* in, int32_t l, std::vector<int32_t>* level, LatInfo* info) {
  const int64_t s0 = in->state_off[l], s1 = in->state_off[l + 1];
  const int64_t e0 = in->arc_off[l], e1 = in->arc_off[l + 1];
  const int32_t ns = (int32_t)(s1 - s0);
  level->assign(ns, 0);
  int32_t prev = 0, maxl = -1;
  for (int64_t e = e0; e < e1; ++e) {
    const int32_t u = in->arc_src[e], v = in->arc_dst[e];
    if (u < prev || u >= ns || v <= u || v >= ns) {
      info->err = "lattice " + std::to_string(l) +
                  ": arcs must be grouped by ascending src and topologically sorted (src < dst)";
      return;
    }
    if (!std::isfinite(in->arc_graph[e]) || !std::isfinite(in->arc_acoustic[e])) {
      info->err = "lattice " + std::to_string(l) + ": non-finite arc weight";
      return;
    }
    prev = u;
    if ((*level)[v] < (*level)[u] + 1) (*level)[v] = (*level)[u] + 1;
  }
  for (int32_t s = 0; s < ns; ++s) maxl = std::max(maxl, (*level)[s]);
  info->nl = maxl + 1;
}

}  // namespace

int pack_and_upload(klu_ctx* c, const klu_lattices* in) {
  const int32_t L = in->num_lattices;
  if (L < 0) {
    set_error("klu_load: negative lattice count");
    return 1;
  }
  const int64_t S = L ? in->state_off[L] - in->state_off[0] : 0;
  const int64_t E = L ? in->arc_off[L] - in->arc_off[0] : 0;
  if (L && (in->state_off[0] != 0 || in->arc_off[0] != 0)) {
    set_error("klu_load: offsets must start at 0");
    return 1;
  }
  if (S >= (int64_t)1 << 31 || E >= (int64_t)1 << 31) {
    set_error("klu_load: batch too large for 32-bit indices; split it");
    return 1;
  }
  std::vector<LatInfo> info(L);
  std::vector<std::vector<int32_t> > levels;  // only kept inside workers
  Staging st;
  st.s_off.resize(L + 1);
  st.e_off.resize(L + 1);
  st.lvl_off.resize(L + 1);
  for (int32_t l = 0; l <= L; ++l) {
    st.s_off[l] = (int32_t)in->state_off[l];
    st.e_off[l] = (int32_t)in->arc_off[l];
  }
  st.in_off.assign(S + 1, 0);
  st.out_off.assign(S + 1, 0);
  st.out_src.resize(E);
  st.out_orig.resize(E);
  st.in2out.resize(E);
  st.in_rec.resize(E);
  st.out_rec.resize(E);
  st.fin_g.resize(S);
  st.fin_a.resize(S);
  st.time.resize(S);
  st.orig.resize(S);
  st.level.resize(S);
  st.band_lo.resize(S);
  st.band_off.assign(S + 1, 0);
  c->h_new2old.resize(S);
  c->h_old2new.resize(S);

  unsigned nthreads = std::max(1u, std::min(std::thread::hardware_concurrency(), 64u));
  if ((int64_t)nthreads > L) nthreads = (unsigned)std::max<int32_t>(1, L);
  // contiguous lattice ranges balanced by arcs
  std::vector<int32_t> range(nthreads + 1, L);
  range[0] = 0;
  {
    int64_t per = (E + nthreads - 1) / nthreads;
    int32_t l = 0;
    for (unsigned t = 1; t < nthreads; ++t) {
      const int64_t target = per * t;
      while (l < L && in->arc_off[l] < target) ++l;
      range[t] = l;
    }
  }

  // ---- phase 1: levels (needs per-lattice level counts before the layout of
  // lvl_start is known) ----
  std::vector<std::vector<int32_t> > lat_level(L);
  {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nthreads; ++t)
      th.emplace_back([&, t]() {
        for (int32_t l = range[t]; l < range[t + 1]; ++l) lattice_levels(in, l, &lat_level[l], &info[l]);
      });
    for (auto& x : th) x.join();
  }
  for (int32_t l = 0; l < L; ++l)
    if (!info[l].err.empty()) {
      set_error("klu_load: " + info[l].err);
      return 1;
    }
  st.lvl_off[0] = 0;
  for (int32_t l = 0; l < L; ++l) st.lvl_off[l + 1] = st.lvl_off[l] + info[l].nl + 1;
  st.lvl_start.resize(st.lvl_off[L]);

  // ---- phase 2: renumber, build both arc orders, times, bands ----
  {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nthreads; ++t)
      th.emplace_back([&, t]() {
        std::vector<int32_t> newid, cnt, times, lo, hi, first_arc, cursor;
        for (int32_t l = range[t]; l < range[t + 1]; ++l) {
          const int64_t s0 = in->state_off[l], e0 = in->arc_off[l];
          const int32_t ns = (int32_t)(in->state_off[l + 1] - s0);
          const int32_t na = (int32_t)(in->arc_off[l + 1] - e0);
          const std::vector<int32_t>& level = lat_level[l];
          LatInfo& li = info[l];
          const int32_t nl = li.nl;
          // counting sort of states by level (stable in input id)
          cnt.assign(nl + 1, 0);
          for (int32_t s = 0; s < ns; ++s) cnt[level[s] + 1]++;
          for (int32_t j = 0; j < nl; ++j) cnt[j + 1] += cnt[j];
          int32_t* lv = st.lvl_start.data() + st.lvl_off[l];
          for (int32_t j = 0; j <= nl; ++j) lv[j] = (int32_t)s0 + cnt[j];
          newid.resize(ns);
          for (int32_t s = 0; s < ns; ++s) newid[s] = cnt[level[s]]++;
          // state times (CompactLatticeStateTimes [ext]) and length bands, input order
          times.assign(ns, -1);
          lo.assign(ns, INT32_MAX);
          hi.assign(ns, -1);
          first_arc.assign(ns + 1, 0);
          if (ns > 0) {
            times[0] = 0;
            lo[0] = 0;
            hi[0] = 0;
          }
          for (int32_t e = 0; e < na; ++e) first_arc[in->arc_src[e0 + e] + 1]++;
          for (int32_t s = 0; s < ns; ++s) first_arc[s + 1] += first_arc[s];
          for (int32_t e = 0; e < na; ++e) {
            const int32_t u = in->arc_src[e0 + e], v = in->arc_dst[e0 + e];
            const int32_t lab = in->arc_label[e0 + e];
            if (times[u] >= 0) {
              const int32_t tv = times[u] + in->arc_dur[e0 + e];
              if (times[v] == -1) times[v] = tv;
              else if (times[v] != tv) li.times_ok = 0;
            }
            if (hi[u] >= 0) {
              const int32_t nz = lab != 0 ? 1 : 0;
              lo[v] = std::min(lo[v], lo[u] + nz);
              hi[v] = std::max(hi[v], hi[u] + nz);
            }
            li.max_label = std::max(li.max_label, lab);
            li.max_span = std::max(li.max_span, in->arc_dur[e0 + e]);
          }
          int32_t utt = -1;
          for (int32_t s = 0; s < ns; ++s) {
            const float fg = in->fin_graph[s0 + s], fa = in->fin_acoustic[s0 + s];
            const bool is_final = !(std::isinf(fg) && std::isinf(fa));
            if (is_final && times[s] >= 0) {
              const int32_t tf = times[s] + (in->fin_dur ? in->fin_dur[s0 + s] : 0);
              utt = std::max(utt, tf);
            }
            if (hi[s] >= 0) li.max_len = std::max(li.max_len, hi[s]);
            li.max_time = std::max(li.max_time, times[s]);
          }
          li.num_frames = utt < 0 ? 0 : utt;
          // per-state arrays in packed order
          for (int32_t s = 0; s < ns; ++s) {
            const int32_t n = (int32_t)s0 + newid[s];
            st.fin_g[n] = in->fin_graph[s0 + s];
            st.fin_a[n] = in->fin_acoustic[s0 + s];
            st.time[n] = times[s];
            st.orig[n] = s;
            st.level[n] = level[s];
            st.band_lo[n] = hi[s] >= 0 ? lo[s] : -1;
            st.band_off[n + 1] = hi[s] >= 0 ? hi[s] - lo[s] + 1 : 0;  // widths; prefix-summed later
            c->h_new2old[n] = s;
            c->h_old2new[s0 + s] = n;
            st.out_off[n + 1] = first_arc[s + 1] - first_arc[s];
            li.max_outdeg = std::max(li.max_outdeg, first_arc[s + 1] - first_arc[s]);
          }
          // local prefix sums (made global after the join)
          // out-order arcs: packed states ascending, stored order within a state
          cursor.assign(ns + 1, 0);  // in-degree histogram by packed dst
          {
            int32_t pos = 0;
            // iterate packed ids: need old id of packed state n -> st.orig
            for (int32_t n = 0; n < ns; ++n) {
              const int32_t s = st.orig[s0 + n];
              for (int32_t e = first_arc[s]; e < first_arc[s + 1]; ++e) {
                const int64_t ge = e0 + e;
                const int32_t d = newid[in->arc_dst[ge]];
                st.out_rec[e0 + pos] = make_int4((int32_t)s0 + d, f2i(in->arc_graph[ge]), f2i(in->arc_acoustic[ge]),
                                                 in->arc_label[ge]);
                st.out_src[e0 + pos] = (int32_t)s0 + n;
                st.out_orig[e0 + pos] = e;
                cursor[d + 1]++;
                ++pos;
                // entry capacity of the arc x frame and arc x length expansions
                if (in->arc_label[ge] != 0) {
                  // frames [t(src), t(dst)) of the arc, inside the utterance
                  const int32_t fa = std::max(times[s], 0), fb = std::min(times[in->arc_dst[ge]], li.num_frames);
                  li.cap_frame += fb > fa ? fb - fa : 0;
                  li.cap_pos += hi[s] >= 0 ? hi[s] - lo[s] + 1 : 0;
                }
              }
            }
          }
          for (int32_t n = 0; n < ns; ++n) {
            st.in_off[s0 + n + 1] = cursor[n + 1];
            li.max_indeg = std::max(li.max_indeg, cursor[n + 1]);
            cursor[n + 1] += cursor[n];
          }
          // in-order arcs: stable counting sort of the out-order by packed dst
          for (int32_t p = 0; p < na; ++p) {
            const int4 r = st.out_rec[e0 + p];
            const int32_t d = r.x - (int32_t)s0;
            st.in2out[e0 + cursor[d]] = (int32_t)(e0 + p);
            st.in_rec[e0 + cursor[d]++] = make_int4(st.out_src[e0 + p], r.y, r.z, r.w);
          }
          lat_level[l] = std::vector<int32_t>();
        }
      });
    for (auto& x : th) x.join();
  }
  // global prefix sums of the per-state counts
  for (int64_t s = 0; s < S; ++s) {
    st.in_off[s + 1] += st.in_off[s];
    st.out_off[s + 1] += st.out_off[s];
  }
  {
    int64_t acc = 0;
    for (int64_t s = 0; s < S; ++s) {
      acc += st.band_off[s + 1];
      st.band_off[s + 1] = acc;
    }
    c->band_total = acc;
    c->h_band_off.resize(L + 1);
    for (int32_t l = 0; l <= L; ++l) c->h_band_off[l] = st.band_off[in->state_off[l]];
  }
  // frame -> arc CSR offsets (the arc x frame expansion of latbin/lattice-to-word-frame-post.cc:110-116
  // as an index structure): per lattice, per frame, the first of the word arcs alive in it; and
  // every arc's start-time key for build_frame_groups
  std::vector<int32_t> fr_base(L + 1, 0);
  std::vector<int64_t> fa_base(L + 1, 0);
  int32_t max_time = 0;
  for (int32_t l = 0; l < L; ++l) {
    fr_base[l + 1] = fr_base[l] + info[l].num_frames + 1;
    fa_base[l + 1] = fa_base[l] + info[l].cap_frame;
    max_time = std::max(max_time, std::max(info[l].max_time, info[l].num_frames));  // = c->max_time below
  }
  std::vector<int64_t> fr_off((size_t)fr_base[L] + 1, 0);
  const uint32_t time_tail = frame_time_tail(max_time);
  std::vector<uint32_t> time_key((size_t)E, time_tail);
  {
    std::vector<std::thread> th;
    for (unsigned t = 0; t < nthreads; ++t)
      th.emplace_back([&, t]() {
        std::vector<int64_t> cur;
        for (int32_t l = range[t]; l < range[t + 1]; ++l) {
          const int32_t T = info[l].num_frames;
          const int64_t e0 = in->arc_off[l], e1 = in->arc_off[l + 1];
          int64_t* fo = fr_off.data() + fr_base[l];
          cur.assign(T + 1, 0);
          for (int64_t p = e0; p < e1; ++p) {
            const int4 r = st.out_rec[p];
            if (r.w == 0) continue;
            const int32_t fa = std::max(st.time[st.out_src[p]], 0), fb = std::min(st.time[r.x], T);
            for (int32_t k = fa; k < fb; ++k) cur[k + 1]++;
            if (fb > fa) time_key[(size_t)p] = (uint32_t)fa;
          }
          for (int32_t k = 0; k < T; ++k) cur[k + 1] += cur[k];
          for (int32_t k = 0; k <= T; ++k) fo[k] = fa_base[l] + cur[k];
        }
      });
    for (auto& x : th) x.join();
  }
  c->h_fr_base = fr_base;
  c->frame_entries = fa_base[L];

  // work queue order: lattices by descending arc count
  st.order.resize(L);
  std::iota(st.order.begin(), st.order.end(), 0);
  std::stable_sort(st.order.begin(), st.order.end(), [&](int32_t a, int32_t b) {
    return (in->arc_off[a + 1] - in->arc_off[a]) > (in->arc_off[b + 1] - in->arc_off[b]);
  });

  // ---- host metadata ----
  c->L = L;
  c->S = S;
  c->E = E;
  c->NL = st.lvl_off[L] - L;
  c->h_s_off.assign(in->state_off, in->state_off + L + 1);
  c->h_e_off.assign(in->arc_off, in->arc_off + L + 1);
  c->h_num_frames.resize(L);
  c->h_maxtime.resize(L);
  c->h_times_ok.resize(L);
  c->h_cap_frame.resize(L);
  c->h_cap_pos.resize(L);
  c->h_maxlen.resize(L);
  c->max_label = c->max_time = c->max_len = c->max_indeg = c->max_outdeg = c->max_states = c->max_span = 0;
  for (int32_t l = 0; l < L; ++l) {
    c->max_span = std::max(c->max_span, info[l].max_span);
    c->h_num_frames[l] = info[l].num_frames;
    c->h_maxtime[l] = std::max(info[l].max_time, info[l].num_frames);
    c->h_times_ok[l] = info[l].times_ok;
    c->h_cap_frame[l] = info[l].cap_frame;
    c->h_cap_pos[l] = info[l].cap_pos;
    c->h_maxlen[l] = info[l].max_len;
    c->max_label = std::max(c->max_label, info[l].max_label);
    c->max_time = std::max(c->max_time, std::max(info[l].max_time, info[l].num_frames));
    c->max_len = std::max(c->max_len, info[l].max_len);
    c->max_indeg = std::max(c->max_indeg, info[l].max_indeg);
    c->max_outdeg = std::max(c->max_outdeg, info[l].max_outdeg);
    c->max_states = std::max<int32_t>(c->max_states, (int32_t)(in->state_off[l + 1] - in->state_off[l]));
  }
  c->avg_deg = S ? (double)E / (double)S : 0.0;

  // ---- upload ----
  auto up = [&](DevBuf& b, const void* src, size_t bytes) -> int {
    KLU_TRY(b.reserve(bytes ? bytes : 16));
    if (bytes) KLU_CUDA(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return 0;
  };
  KLU_TRY(up(c->d_s_off, st.s_off.data(), st.s_off.size() * 4));
  KLU_TRY(up(c->d_e_off, st.e_off.data(), st.e_off.size() * 4));
  KLU_TRY(up(c->d_lvl_off, st.lvl_off.data(), st.lvl_off.size() * 4));
  KLU_TRY(up(c->d_lvl_start, st.lvl_start.data(), st.lvl_start.size() * 4));
  KLU_TRY(up(c->d_in_rec, st.in_rec.data(), st.in_rec.size() * sizeof(int4)));
  KLU_TRY(up(c->d_out_rec, st.out_rec.data(), st.out_rec.size() * sizeof(int4)));
  KLU_TRY(up(c->d_in_off, st.in_off.data(), st.in_off.size() * 4));
  KLU_TRY(up(c->d_out_off, st.out_off.data(), st.out_off.size() * 4));
  KLU_TRY(up(c->d_out_src, st.out_src.data(), st.out_src.size() * 4));
  KLU_TRY(up(c->d_out_orig, st.out_orig.data(), st.out_orig.size() * 4));
  KLU_TRY(up(c->d_in2out, st.in2out.data(), st.in2out.size() * 4));
  KLU_TRY(up(c->d_fin_g, st.fin_g.data(), st.fin_g.size() * 4));
  KLU_TRY(up(c->d_fin_a, st.fin_a.data(), st.fin_a.size() * 4));
  KLU_TRY(up(c->d_time, st.time.data(), st.time.size() * 4));
  KLU_TRY(up(c->d_orig, st.orig.data(), st.orig.size() * 4));
  KLU_TRY(up(c->d_old2new, c->h_old2new.data(), c->h_old2new.size() * 4));
  KLU_TRY(up(c->d_level, st.level.data(), st.level.size() * 4));
  KLU_TRY(up(c->d_band_lo, st.band_lo.data(), st.band_lo.size() * 4));
  KLU_TRY(up(c->d_band_off, st.band_off.data(), st.band_off.size() * 8));
  KLU_TRY(up(c->d_order, st.order.data(), st.order.size() * 4));
  KLU_TRY(up(c->d_fr_base, fr_base.data(), fr_base.size() * 4));
  KLU_TRY(up(c->d_fr_off, fr_off.data(), fr_off.size() * 8));
  {
    uint32_t* keys = nullptr;
    KLU_TRY(reserve_frame_time_keys(c, &keys));  // after c->frame_entries and c->E are set
    if (E) KLU_CUDA(cudaMemcpyAsync(keys, time_key.data(), time_key.size() * 4, cudaMemcpyHostToDevice, c->stream));
  }
  KLU_CUDA(cudaStreamSynchronize(c->stream));  // staging vectors die here
  return build_frame_groups(c);
}

}  // namespace klu
