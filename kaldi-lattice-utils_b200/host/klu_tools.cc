// klu_tools.cc -- the seven drop-in command-line tools.  One source, compiled
// once per tool with -DKLU_TOOL=<enum klu_tool>; each keeps the reference
// binary's name, flags, positional arguments, output format, stderr logging
// style and exit codes (SURVEY.md 8b), and hands the per-lattice work of the
// reference's functor body to the GPU engine through include/klu.h in batches:
//
//   lattice-word-index-position   kwsbin2/lattice-word-index-position.cc:208-297
//   lattice-word-index-segment    kwsbin2/lattice-word-index-segment.cc:194-282
//   lattice-word-index-utterance  kwsbin2/lattice-word-index-utterance.cc:194-328
//   lattice-char-index-position   kwsbin2/lattice-char-index-position.cc:303-409
//   lattice-to-word-frame-post    latbin/lattice-to-word-frame-post.cc:29-147
//   lattice-prune-dyn-beam        latbin/lattice-prune-dyn-beam.cc:97-214
//   lattice-best-path2            latbin/lattice-best-path2.cc:29-221
//   lattice-to-word-position-post latbin/lattice-to-word-position-post.cc:28-147 (SURVEY.md 8f)
//   lattice-char-index-segment    kwsbin2/lattice-char-index-segment.cc:249-349 (SURVEY.md 8f)
//   lattice-to-transcript-length-dist latbin/lattice-to-transcript-length-dist.cc:28-131 (SURVEY.md 8f)
//   lattice-char-index-utterance  (no reference binary; the flags of lattice-char-index-segment)
//
// Lattices are independent, so the reader fills a batch (KLU_BATCH_ARCS arcs,
// default 32M), the batch is packed/uploaded/processed, and entries are written
// in input order -- the TaskSequencer contract (P9); parsing, GPU work and writing
// of successive batches overlap (class Pipeline).  --num-threads is accepted
// and ignored.  KLU_DEVICE selects the GPU (default 0), KLU_DEVICES=a,b,... several contexts.
#include <limits.h>
#include <malloc.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <exception>
#include <memory>
#include <mutex>
#include <set>
#include <thread>

#include "kaldi_io.h"
#include "klu.h"

#ifndef KLU_TOOL
#error "compile with -DKLU_TOOL=<tool id>"
#endif

using namespace kio;

namespace {

#define KLU_CHECK(call)                                          \
  do {                                                           \
    if ((call) != 0) KIO_ERR("GPU engine: " << klu_last_error()); \
  } while (0)

// The tools close a batch at this many lattices whatever their size (archives of tiny lattices:
// bounds the per-lattice host metadata of a batch); the library itself has no such limit.
#if KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
// The character tools keep every same-group sub-path of a batch in device memory at once (a trie
// whose frontier can grow by the branching factor per character): small batches bound that
// (256 c5 lattices: ~1.6e8 candidates at the deepest level, a few GB).
constexpr size_t kMaxBatchLattices = 256;
#else
constexpr size_t kMaxBatchLattices = (size_t)1 << 20;
#endif

struct Batch {
  std::vector<CompactLat> lats;
  std::vector<int64_t> state_off{0}, arc_off{0};
  std::vector<int32_t> src, dst, label, dur, fin_dur;
  std::vector<float> graph, acoustic, fin_graph, fin_acoustic;
  int64_t arcs() const { return arc_off.back(); }
  void Add(CompactLat&& l, bool keep_lattice) {
    src.insert(src.end(), l.src.begin(), l.src.end());
    dst.insert(dst.end(), l.dst.begin(), l.dst.end());
    label.insert(label.end(), l.label.begin(), l.label.end());
    dur.insert(dur.end(), l.dur.begin(), l.dur.end());
    graph.insert(graph.end(), l.graph.begin(), l.graph.end());
    acoustic.insert(acoustic.end(), l.acoustic.begin(), l.acoustic.end());
    fin_graph.insert(fin_graph.end(), l.fin_graph.begin(), l.fin_graph.end());
    fin_acoustic.insert(fin_acoustic.end(), l.fin_acoustic.begin(), l.fin_acoustic.end());
    fin_dur.insert(fin_dur.end(), l.fin_dur.begin(), l.fin_dur.end());
    state_off.push_back(state_off.back() + l.nstates);
    arc_off.push_back(arc_off.back() + (int64_t)l.src.size());
    if (!keep_lattice) {  // only prune-dyn-beam writes lattices back
      CompactLat slim;
      slim.key = l.key;
      slim.nstates = l.nstates;
      lats.push_back(std::move(slim));
    } else {
      lats.push_back(std::move(l));
    }
  }
  // A block of lattices at once: the arrays grow once and the lattices are copied in by
  // several threads (SequentialCompactLatticeReader::ReadBlock delivers such blocks).
  void AddBlock(std::vector<CompactLat>* block, bool keep_lattice) {
    const size_t n0 = lats.size(), nb = block->size();
    for (const CompactLat& l : *block) {
      state_off.push_back(state_off.back() + l.nstates);
      arc_off.push_back(arc_off.back() + (int64_t)l.src.size());
    }
    const size_t E = (size_t)arc_off.back(), S = (size_t)state_off.back();
    src.resize(E), dst.resize(E), label.resize(E), dur.resize(E), graph.resize(E), acoustic.resize(E);
    fin_graph.resize(S), fin_acoustic.resize(S), fin_dur.resize(S);
    lats.resize(n0 + nb);
    ParallelFor(nb, [&](size_t i) {
      CompactLat& l = (*block)[i];
      const size_t e = (size_t)arc_off[n0 + i], s = (size_t)state_off[n0 + i], na = l.src.size();
      if (na) {
        memcpy(&src[e], l.src.data(), 4 * na), memcpy(&dst[e], l.dst.data(), 4 * na);
        memcpy(&label[e], l.label.data(), 4 * na), memcpy(&dur[e], l.dur.data(), 4 * na);
        memcpy(&graph[e], l.graph.data(), 4 * na), memcpy(&acoustic[e], l.acoustic.data(), 4 * na);
      }
      if (l.nstates) {
        memcpy(&fin_graph[s], l.fin_graph.data(), 4 * (size_t)l.nstates);
        memcpy(&fin_acoustic[s], l.fin_acoustic.data(), 4 * (size_t)l.nstates);
        memcpy(&fin_dur[s], l.fin_dur.data(), 4 * (size_t)l.nstates);
      }
      if (keep_lattice) {
        lats[n0 + i] = std::move(l);
      } else {
        lats[n0 + i].key = l.key;
        lats[n0 + i].nstates = l.nstates;
      }
    });
    block->clear();
  }
  // What goes over PCIe: per-state arc counts instead of per-arc sources (the arcs are grouped by
  // source state, as OpenFst stores them), durations as bytes and destinations as 16-bit distances
  // from the source when they all fit (klu_lattices.state_num_arcs / arc_dur_u8 /
  // arc_dst_delta_u16), labels as 16-bit words (arc_label_u16): 13 instead of 24 bytes per arc.
  // Built once per batch on the I/O threads.
  mutable std::vector<int32_t> num_arcs_;
  mutable std::vector<uint8_t> dur8_;
  mutable std::vector<uint16_t> delta16_, label16_;
  klu_lattices View() const {
    klu_lattices v;
    memset(&v, 0, sizeof(v));
    v.num_lattices = (int32_t)lats.size();
    v.state_off = state_off.data();
    v.arc_off = arc_off.data();
    v.arc_src = src.data();
    v.arc_dst = dst.data();
    v.arc_label = label.data();
    v.arc_dur = dur.data();
    v.arc_graph = graph.data();
    v.arc_acoustic = acoustic.data();
    v.fin_graph = fin_graph.data();
    v.fin_acoustic = fin_acoustic.data();
    v.fin_dur = fin_dur.data();
    const size_t E = src.size(), S = fin_graph.size(), nl = lats.size();
    num_arcs_.assign(S, 0);
    dur8_.resize(E);
    delta16_.resize(E);
    label16_.resize(E);
    std::atomic<int> dur_ok(1), delta_ok(1), grouped(1), label_ok(1);
    ParallelFor(nl, [&](size_t l) {
      const size_t e0 = (size_t)arc_off[l], e1 = (size_t)arc_off[l + 1], s0 = (size_t)state_off[l];
      const int32_t ns = (int32_t)(state_off[l + 1] - state_off[l]);
      bool d_ok = true, t_ok = true, g_ok = true, l_ok = true;
      for (size_t e = e0; e < e1; ++e) {
        const int32_t u = src[e], dd = dst[e] - u, du = dur[e], lb = label[e];
        if (u < 0 || u >= ns || (e > e0 && src[e - 1] > u)) { g_ok = false; break; }
        ++num_arcs_[s0 + (size_t)u];
        if (du < 0 || du > 255) d_ok = false;
        if (dd < 0 || dd > 65535) t_ok = false;
        if (lb < 0 || lb > 65535) l_ok = false;
        dur8_[e] = (uint8_t)du;
        delta16_[e] = (uint16_t)dd;
        label16_[e] = (uint16_t)lb;
      }
      if (!l_ok) label_ok = 0;
      if (!d_ok) dur_ok = 0;
      if (!t_ok) delta_ok = 0;
      if (!g_ok) grouped = 0;
    });
    if (grouped) {  // (otherwise klu_load reports the layout error from the plain arrays)
      v.arc_src = nullptr;
      v.state_num_arcs = num_arcs_.data();
      if (dur_ok) {
        v.arc_dur = nullptr;
        v.arc_dur_u8 = dur8_.data();
      }
      if (delta_ok) {
        v.arc_dst = nullptr;
        v.arc_dst_delta_u16 = delta16_.data();
      }
      if (label_ok) {
        v.arc_label = nullptr;
        v.arc_label_u16 = label16_.data();
      }
    }
    return v;
  }
};

struct ToolState {
  std::vector<klu_ctx*> ctxs;  // one per GPU (KLU_DEVICES)
  klu_opts opts;
  std::vector<int32_t> include, exclude, group_labels, group_ids, inc_groups, del_groups;
  TableWriter* writer = nullptr;
  double total_cost = 0.0;       // best-path2
  int64_t total_frames = 0;
  size_t num_lattices = 0;
  double sec_read = 0.0, sec_wait = 0.0, sec_gpu = 0.0, sec_emit = 0.0;  // KLU_TRACE summary
};

[[maybe_unused]] void WriteTupleSep(std::ostream& os, bool binary, size_t i, size_t n) {
  if (!binary && i + 1 < n) os.rdbuf()->sputn("; ", 2);
}

// Everything klu_fetch_* returns for one batch (which fields are used depends on the tool).
struct Results {
  std::vector<int64_t> off, coff;
  std::vector<int32_t> i0, i1, i2, i3, chars, smap;
  std::vector<double> d0, beams;
  std::vector<float> f0, f1, f2, f3;
  std::string error;
  double sec = 0.0;
};

// GPU part of a batch: pack + upload, run the tool, bring the results to the host.
// Runs on the worker thread that owns `ctx` (one context per GPU).
void ComputeBatch(klu_ctx* ctx, const klu_opts* opts, const Batch* b, Results* r) {
  try {
    const int32_t L = (int32_t)b->lats.size();
    const auto t0 = std::chrono::steady_clock::now();
    klu_lattices view = b->View();
    KLU_CHECK(klu_load(ctx, &view));
    KLU_CHECK(klu_run(ctx, KLU_TOOL, opts));
    r->off.resize(L + 1);
    KLU_CHECK(klu_result_offsets(ctx, r->off.data()));
    const size_t n = (size_t)r->off[L];
#if KLU_TOOL == 0 /* KLU_SEGMENT */
    r->i0.resize(n), r->i1.resize(n), r->i2.resize(n), r->d0.resize(n);
    KLU_CHECK(klu_fetch_segment(ctx, r->i0.data(), r->i1.data(), r->i2.data(), r->d0.data()));
#elif KLU_TOOL == 1 /* KLU_POSITION */
    r->i0.resize(n), r->i1.resize(n), r->i2.resize(n), r->i3.resize(n), r->d0.resize(n);
    KLU_CHECK(klu_fetch_position(ctx, r->i0.data(), r->i1.data(), r->i2.data(), r->i3.data(), r->d0.data()));
#elif KLU_TOOL == 2 /* KLU_UTTERANCE */
    r->i0.resize(n), r->d0.resize(n);
    KLU_CHECK(klu_fetch_utterance(ctx, r->i0.data(), r->d0.data()));
#elif KLU_TOOL == 6 /* KLU_CHAR_POSITION */
    int64_t total_chars = 0;
    KLU_CHECK(klu_result_char_sizes(ctx, &total_chars));
    r->coff.resize(n + 1), r->chars.resize((size_t)total_chars);
    r->i1.resize(n), r->i2.resize(n), r->i3.resize(n), r->d0.resize(n);
    KLU_CHECK(klu_fetch_char_position(ctx, r->coff.data(), r->chars.data(), r->i1.data(), r->i2.data(), r->i3.data(),
                                      r->d0.data()));
#elif KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */
    int64_t total_chars = 0;
    KLU_CHECK(klu_result_char_sizes(ctx, &total_chars));
    r->coff.resize(n + 1), r->chars.resize((size_t)total_chars);
    r->i2.resize(n), r->i3.resize(n), r->d0.resize(n);
    KLU_CHECK(klu_fetch_char_segment(ctx, r->coff.data(), r->chars.data(), r->i2.data(), r->i3.data(), r->d0.data()));
#elif KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
    int64_t total_chars = 0;
    KLU_CHECK(klu_result_char_sizes(ctx, &total_chars));
    r->coff.resize(n + 1), r->chars.resize((size_t)total_chars);
    r->d0.resize(n);
    KLU_CHECK(klu_fetch_char_utterance(ctx, r->coff.data(), r->chars.data(), r->d0.data()));
#elif KLU_TOOL == 3 /* KLU_FRAME_POST */
    // rows without the per-row frame column (a third of the download); the writer below shares
    // its loop with the position-post / length-dist tools, which carry one, so it is rebuilt here
    r->i0.resize(L), r->i1.resize(n), r->i2.resize(n), r->f0.resize(n);
    KLU_CHECK(klu_fetch_frame_post_csr(ctx, r->i0.data(), nullptr, nullptr, nullptr));  // frame counts
    {
      std::vector<int64_t> slot((size_t)L + 1, 0);
      for (int32_t l = 0; l < L; ++l) slot[l + 1] = slot[l] + r->i0[l] + 1;
      std::vector<int64_t> fo((size_t)slot[L]);
      KLU_CHECK(klu_fetch_frame_post_csr(ctx, r->i0.data(), fo.data(), r->i2.data(), r->f0.data()));
      ParallelFor((size_t)L, [&](size_t l) {
        const int64_t* f = fo.data() + slot[l];
        const size_t a = (size_t)r->off[l];
        for (int32_t k = 0; k < r->i0[l]; ++k)
          for (int64_t i = f[k]; i < f[k + 1]; ++i) r->i1[a + (size_t)i] = k;
      });
    }
#elif KLU_TOOL == 10 /* KLU_LENGTH_DIST */
    // one Posterior frame per lattice (latbin/lattice-to-transcript-length-dist.cc:111)
    r->i0.assign(L, 1), r->i1.assign(n, 0), r->i2.resize(n), r->f0.resize(n);
    KLU_CHECK(klu_fetch_length_dist(ctx, r->i2.data(), r->f0.data()));
#elif KLU_TOOL == 8 /* KLU_POSITION_POST */
    r->i0.resize(L), r->i1.resize(n), r->i2.resize(n), r->f0.resize(n);
    KLU_CHECK(klu_fetch_position_post(ctx, r->i0.data(), r->i1.data(), r->i2.data(), r->f0.data()));
#elif KLU_TOOL == 5 /* KLU_BEST_PATH2 */
    r->i0.resize(n), r->i1.resize(L), r->f0.resize(L);
    KLU_CHECK(klu_fetch_best_path2(ctx, r->i0.data(), r->f0.data(), r->i1.data()));
#elif KLU_TOOL == 4 /* KLU_PRUNE_DYN_BEAM */ || KLU_TOOL == 11 /* KLU_PRUNE_ARCS */
    const size_t S = (size_t)b->state_off.back();
    r->i0.resize(n), r->i1.resize(n), r->i2.resize(n), r->smap.resize(S);
    r->f0.resize(n), r->f1.resize(n), r->f2.resize(S), r->f3.resize(S), r->beams.resize(2 * (size_t)L);
    KLU_CHECK(klu_fetch_prune(ctx, r->i0.data(), r->i1.data(), r->i2.data(), r->f0.data(), r->f1.data(), r->smap.data(),
                              r->f2.data(), r->f3.data(), r->beams.data()));
#endif
    r->sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  } catch (const std::exception& e) {
    r->error = e.what();
  }
}

// Host part: writes the batch's entries in input order (TaskSequencer contract, P9).
void EmitBatch(ToolState* st, Batch* b, Results* r) {
  if (!r->error.empty()) throw std::runtime_error(r->error);
  const int32_t L = (int32_t)b->lats.size();
  const std::vector<int64_t>& off = r->off;
  TableWriter& w = *st->writer;
  const bool bin = w.IsOpen() ? w.binary() : false;
#if KLU_TOOL == 0 /* KLU_SEGMENT */
  for (int32_t l = 0; l < L; ++l) {
    std::ostream& os = w.Begin(b->lats[l].key);
    const size_t a = (size_t)off[l], e = (size_t)off[l + 1];
    if (bin) {
      os.put('\0');
      os.put('B');
      WriteBasicInt32(os, true, (int32_t)(e - a));
    }
    for (size_t i = a; i < e; ++i) {
      WriteBasicInt32(os, bin, r->i0[i]);
      WriteBasicInt32(os, bin, r->i1[i]);
      WriteBasicInt32(os, bin, r->i2[i]);
      WriteBasicDouble(os, bin, r->d0[i]);
      WriteTupleSep(os, bin, i - a, e - a);
    }
    if (!bin) os << '\n';
    w.End();
  }
#elif KLU_TOOL == 1 /* KLU_POSITION */
  for (int32_t l = 0; l < L; ++l) {
    std::ostream& os = w.Begin(b->lats[l].key);
    const size_t a = (size_t)off[l], e = (size_t)off[l + 1];
    if (bin) {
      os.put('\0');
      os.put('B');
      WriteBasicInt32(os, true, (int32_t)(e - a));
    }
    for (size_t i = a; i < e; ++i) {
      WriteBasicInt32(os, bin, r->i0[i]);
      WriteBasicInt32(os, bin, r->i1[i]);
      WriteBasicInt32(os, bin, r->i2[i]);
      WriteBasicInt32(os, bin, r->i3[i]);
      WriteBasicDouble(os, bin, r->d0[i]);
      WriteTupleSep(os, bin, i - a, e - a);
    }
    if (!bin) os << '\n';
    w.End();
  }
#elif KLU_TOOL == 2 /* KLU_UTTERANCE */
  for (int32_t l = 0; l < L; ++l) {
    std::ostream& os = w.Begin(b->lats[l].key);
    const size_t a = (size_t)off[l], e = (size_t)off[l + 1];
    if (bin) {
      os.put('\0');
      os.put('B');
      WriteBasicInt32(os, true, (int32_t)(e - a));
    }
    for (size_t i = a; i < e; ++i) {
      WriteBasicInt32(os, bin, r->i0[i]);
      WriteBasicDouble(os, bin, r->d0[i]);
      WriteTupleSep(os, bin, i - a, e - a);
    }
    if (!bin) os << '\n';
    w.End();
  }
#elif KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
  for (int32_t l = 0; l < L; ++l) {
    std::ostream& os = w.Begin(b->lats[l].key);
    const size_t a = (size_t)off[l], e = (size_t)off[l + 1];
    if (bin) {
      os.put('\0');
      os.put('B');
      WriteBasicInt32(os, true, (int32_t)(e - a));
    }
    for (size_t i = a; i < e; ++i) {
      std::string tok;
      for (int64_t k = r->coff[i]; k < r->coff[i + 1]; ++k) {
        if (k > r->coff[i]) tok += "_";
        tok += std::to_string(r->chars[(size_t)k]);
      }
      WriteToken(os, bin, tok);
#if KLU_TOOL == 6 /* KLU_CHAR_POSITION */
      WriteBasicInt32(os, bin, r->i1[i]);
#endif
#if KLU_TOOL != 12 /* KLU_CHAR_UTTERANCE: (string, logp) */
      WriteBasicInt32(os, bin, r->i2[i]);
      WriteBasicInt32(os, bin, r->i3[i]);
#endif
      WriteBasicDouble(os, bin, r->d0[i]);
      WriteTupleSep(os, bin, i - a, e - a);
    }
    if (!bin) os << '\n';
    w.End();
  }
#elif KLU_TOOL == 3 /* KLU_FRAME_POST */ || KLU_TOOL == 8 /* KLU_POSITION_POST */ || KLU_TOOL == 10 /* KLU_LENGTH_DIST */
  const std::vector<int32_t>&nf = r->i0, &frame = r->i1, &word = r->i2;
  const std::vector<float>& lp = r->f0;
  // [ext] PosteriorHolder: text "[ lab p lab p ] [ ... ] \n"; binary "\0B" +
  // int32 #frames, per frame int32 n then n x (int32, float), every number behind its
  // size byte.  Binary entries are laid out in memory, several lattices at a time on as
  // many threads, and written with one call each.
  if (bin && w.IsOpen()) {
    std::vector<std::string> bufs((size_t)L);
    ParallelFor((size_t)L, [&](size_t l) {
      const size_t a = (size_t)off[l], e = (size_t)off[l + 1];
      std::string& buf = bufs[l];
      buf.resize(2 + 5 + 5 * (size_t)nf[l] + 10 * (e - a));
      char* q = &buf[0];
      auto put32 = [&q](const void* v) {
        *q++ = 4;
        memcpy(q, v, 4);
        q += 4;
      };
      *q++ = '\0';
      *q++ = 'B';
      put32(&nf[l]);
      size_t i = a;
      for (int32_t k = 0; k < nf[l]; ++k) {
        size_t j = i;
        while (j < e && frame[j] == k) ++j;
        const int32_t n = (int32_t)(j - i);
        put32(&n);
        for (; i < j; ++i) {
          put32(&word[i]);
          put32(&lp[i]);
        }
      }
      buf.resize((size_t)(q - &buf[0]));  // rows outside 0..nf-1 (there are none) would have been skipped
    });
    for (int32_t l = 0; l < L; ++l) {
      std::ostream& os = w.Begin(b->lats[l].key);
      os.write(bufs[l].data(), (std::streamsize)bufs[l].size());
      w.End();
    }
  }
  for (int32_t l = 0; l < L && !(bin && w.IsOpen()); ++l) {
    std::ostream& os = w.Begin(b->lats[l].key);
    size_t i = (size_t)off[l];
    const size_t e = (size_t)off[l + 1];
    if (bin) {
      os.put('\0');
      os.put('B');
      WriteBasicInt32(os, true, nf[l]);
    }
    for (int32_t k = 0; k < nf[l]; ++k) {
      size_t j = i;
      while (j < e && frame[j] == k) ++j;
      if (bin) {
        WriteBasicInt32(os, true, (int32_t)(j - i));
        for (; i < j; ++i) {
          WriteBasicInt32(os, true, word[i]);
          WriteBasicFloat(os, true, lp[i]);
        }
      } else {
        os << "[ ";
        for (; i < j; ++i) {
          os << word[i] << ' ';
          WriteKaldiFloat(os, lp[i]);
          os << ' ';
        }
        os << "] ";
      }
    }
    if (!bin) os << '\n';
    w.End();
  }
#elif KLU_TOOL == 5 /* KLU_BEST_PATH2 */
  const std::vector<int32_t>&lab = r->i0, &nf = r->i1;
  const std::vector<float>& cost = r->f0;
  for (int32_t l = 0; l < L; ++l) {
    if (w.IsOpen()) {
      std::ostream& os = w.Begin(b->lats[l].key);
      const size_t a = (size_t)off[l], e = (size_t)off[l + 1];
      if (bin) {  // [ext] BasicVectorHolder<int32>
        os.put('\0');
        os.put('B');
        WriteBasicInt32(os, true, (int32_t)(e - a));
      }
      for (size_t i = a; i < e; ++i) WriteBasicInt32(os, bin, lab[i]);
      if (!bin) os << '\n';
      w.End();
    }
    st->total_cost += cost[l];
    st->total_frames += nf[l];
    KIO_LOG("For utterance " << b->lats[l].key << ", best cost is " << cost[l] << " over " << nf[l] << " frames.");
  }
#elif KLU_TOOL == 4 /* KLU_PRUNE_DYN_BEAM */ || KLU_TOOL == 11 /* KLU_PRUNE_ARCS */
  const std::vector<int32_t>&ai = r->i0, &ns = r->i1, &nd = r->i2, &smap = r->smap;
  const std::vector<float>&g = r->f0, &a = r->f1, &fg = r->f2, &fa = r->f3;
  const std::vector<double>& beams = r->beams;
  for (int32_t l = 0; l < L; ++l) {
    const CompactLat& in = b->lats[l];
    const size_t s0 = (size_t)b->state_off[l];
    CompactLat out;
    out.key = in.key;
    int32_t nstates = 0;
    for (int32_t s = 0; s < in.nstates; ++s) nstates = std::max(nstates, smap[s0 + s] + 1);
    out.nstates = nstates;
    const float inf = std::numeric_limits<float>::infinity();
    out.fin_graph.assign(nstates, inf);
    out.fin_acoustic.assign(nstates, inf);
    out.fin_dur.assign(nstates, 0);
    out.fin_tids.assign(nstates, TidString());
    for (int32_t s = 0; s < in.nstates; ++s) {
      const int32_t m = smap[s0 + s];
      if (m < 0) continue;
      out.fin_graph[m] = fg[s0 + s];
      out.fin_acoustic[m] = fa[s0 + s];
      if (!(std::isinf(fg[s0 + s]) && std::isinf(fa[s0 + s]))) out.fin_tids[m] = in.fin_tids[s];
    }
    for (size_t i = (size_t)off[l]; i < (size_t)off[l + 1]; ++i) {
      out.src.push_back(ns[i]);
      out.dst.push_back(nd[i]);
      out.label.push_back(in.label[ai[i]]);
      out.dur.push_back(in.dur[ai[i]]);
      out.graph.push_back(g[i]);
      out.acoustic.push_back(a[i]);
      out.tids.push_back(in.tids[ai[i]]);
    }
    std::ostream& os = w.Begin(in.key);
    WriteCompactLattice(os, bin, out);
    w.End();
    const int64_t oa = (int64_t)in.src.size(), na = off[l + 1] - off[l];
#if KLU_TOOL == 11 /* KLU_PRUNE_ARCS */
    (void)beams;
    KIO_LOG("Lattice " << in.key << " pruned #states from " << in.nstates << " to " << nstates << " and #arcs from "
                       << oa << " to " << na);  // latbin/lattice-prune-arcs.cc:161-164
    continue;
#endif
    if (in.nstates == nstates && oa == na) {
      KIO_LOG("Lattice " << in.key << " was not pruned (beam = " << beams[2 * l] << ", # states = " << in.nstates
                         << ", # arcs = " << oa << ")");
    } else {
      KIO_LOG("Lattice " << in.key << " pruned #states from " << in.nstates << " to " << nstates << " and #arcs from "
                         << oa << " to " << na << " (beam reduced from " << beams[2 * l] << " to " << beams[2 * l + 1]
                         << ")");
    }
  }
#endif
  st->num_lattices += (size_t)L;
  KIO_VLOG(1, "Batch of " << L << " lattices (" << b->arcs() << " arcs): done in " << r->sec << " seconds.");
}

// Reading, GPU work and writing overlap: the main thread parses lattices into batches,
// one worker thread per context (KLU_DEVICES; a GPU may be listed more than once) packs,
// runs and fetches them, and a writer thread emits the results strictly in input order
// (the TaskSequencer contract, P9).  At most contexts + 2 batches exist at a time.
class Pipeline {
 public:
  explicit Pipeline(ToolState* st) : st_(st) {
    for (klu_ctx* ctx : st->ctxs) workers_.emplace_back(&Pipeline::Work, this, ctx);
    writer_ = std::thread(&Pipeline::Write, this);
  }
  ~Pipeline() { Shutdown(); }

  // Hands a batch over; blocks while the pipeline is full.  False once a stage has failed.
  bool Submit(Batch&& b) {
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [&] { return abort_ || jobs_.size() < st_->ctxs.size() + 2; });
    if (abort_) return false;
    jobs_.emplace_back(new Job());
    jobs_.back()->b = std::move(b);
    cv_.notify_all();
    return true;
  }

  // Waits for everything submitted to be written; rethrows the first failure of any stage.
  void Finish() {
    Shutdown();
    if (failure_) std::rethrow_exception(failure_);
  }

 private:
  struct Job {
    Batch b;
    Results r;
    bool done = false;
  };

  void Shutdown() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      closing_ = true;
      cv_.notify_all();
    }
    for (auto& t : workers_)
      if (t.joinable()) t.join();
    if (writer_.joinable()) writer_.join();
  }

  void Fail() {
    std::lock_guard<std::mutex> lk(mu_);
    if (!failure_) failure_ = std::current_exception();
    abort_ = true;
    cv_.notify_all();
  }

  void Work(klu_ctx* ctx) {
    for (;;) {
      Job* job = nullptr;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return abort_ || claimed_ < jobs_.size() || closing_; });
        if (abort_ || claimed_ >= jobs_.size()) return;  // closing and nothing left to claim
        job = jobs_[claimed_++].get();
      }
      ComputeBatch(ctx, &st_->opts, &job->b, &job->r);  // failures travel in r.error to the writer
      {
        std::lock_guard<std::mutex> lk(mu_);
        job->done = true;
        cv_.notify_all();
      }
    }
  }

  void Write() {
    try {
      for (;;) {
        std::unique_ptr<Job> job;
        {
          std::unique_lock<std::mutex> lk(mu_);
          cv_.wait(lk, [&] { return abort_ || (!jobs_.empty() && jobs_.front()->done) || (closing_ && jobs_.empty()); });
          if (abort_ || jobs_.empty()) return;
          job = std::move(jobs_.front());
          jobs_.pop_front();
          --claimed_;
          cv_.notify_all();
        }
        const auto t0 = std::chrono::steady_clock::now();
        st_->sec_gpu += job->r.sec;
        EmitBatch(st_, &job->b, &job->r);
        st_->sec_emit += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
      }
    } catch (...) {
      Fail();
    }
  }

  ToolState* st_;
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<std::unique_ptr<Job>> jobs_;  // input order; the front is the next one to write
  size_t claimed_ = 0;                     // jobs_[0 .. claimed_) have been taken by a worker
  bool closing_ = false, abort_ = false;
  std::exception_ptr failure_;
  std::vector<std::thread> workers_;
  std::thread writer_;
};

}  // namespace

int main(int argc, char* argv[]) {
  // the parser threads allocate and free MB-sized arrays all the time: keep those in the
  // heap (no mmap / munmap and fresh page faults per array)
  mallopt(M_MMAP_THRESHOLD, 1 << 30);
  mallopt(M_TRIM_THRESHOLD, 1 << 30);
#if KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
  const int kErrorCode = 1;  // kwsbin2/lattice-char-index-position.cc:405-408
#else
  const int kErrorCode = -1;  // e.g. kwsbin2/lattice-word-index-position.cc:293-296
#endif
  try {
    ToolState st;
    klu_opts_default(&st.opts);
    float beam = std::numeric_limits<float>::infinity();
    float acoustic_scale = 1.0f, graph_scale = 1.0f, insertion_penalty = 0.0f;
    std::string exclude_str, include_str, other_groups_str;
    int32_t num_threads = 1, num_threads_total = -1;
    (void)num_threads;
    (void)num_threads_total;
#if KLU_TOOL == 1 /* KLU_POSITION */
    const char* usage =
        "This tool creates a positional inverted index of the given lattices, in the traditional meaning of "
        "\"position\" in the context of search engines. That is, the probability that a word appears at some "
        "position within the transcription, for all possible transcriptions of the utterance.\n\n"
        "Usage: lattice-word-index-position [options] lat-rspecifier index-wspecifier\n"
        " e.g.: lattice-word-index-position --acoustic-scale=0.1 ark:1.lats ark:1.word.pos.index\n";
#elif KLU_TOOL == 0 /* KLU_SEGMENT */
    const char* usage =
        "This tool creates a positional inverted index of the given lattices, where the score of each word in a "
        "segment is the probability that the word occurs in any of the transcriptions of the utterance at that "
        "specific time segment.\n\n"
        "Usage: lattice-word-index-segment [options] lat-rspecifier index-wspecifier\n"
        " e.g.: lattice-word-index-segment --acoustic-scale=0.1 ark:1.lats ark:1.word.seg.index\n";
#elif KLU_TOOL == 2 /* KLU_UTTERANCE */
    const char* usage =
        "This tool creates an inverted index of the given lattices, where the score of each word is the "
        "probability that the word occurs in any of the transcriptions of the utterance at least once.\n\n"
        "Usage: lattice-word-index-utterance [options] lat-rspecifier index-wspecifier\n"
        " e.g.: lattice-word-index-utterance --acoustic-scale=0.1 ark:1.lats ark:1.word.utt.index\n";
#elif KLU_TOOL == 6 /* KLU_CHAR_POSITION */
    const char* usage =
        "Build a position-level word index from character lattices. Characters are grouped (whitespace group, "
        "optional other groups, default group) and every maximal sub-path of same-group arcs is a pseudo-word.\n\n"
        "Usage: lattice-char-index-position [options] separator-symbols lat-rspecifier index-wspecifier\n"
        " e.g.: lattice-char-index-position \"3 4\" ark:1.lats ark:1.index\n";
#elif KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */
    const char* usage =
        "Build a segment-level word index from character lattices. Characters are grouped (whitespace group, "
        "optional other groups, default group) and every maximal sub-path of same-group arcs is a pseudo-word.\n\n"
        "Usage: lattice-char-index-segment [options] separator-symbols lat-rspecifier index-wspecifier\n"
        " e.g.: lattice-char-index-segment \"3 4\" ark:1.lats ark:1.index\n";
#elif KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
    const char* usage =
        "Build an utterance-level word index from character lattices: the score of each pseudo-word is the "
        "probability that it occurs at least once in the line. Characters are grouped (whitespace group, optional "
        "other groups, default group) and every maximal sub-path of same-group arcs is a pseudo-word.\n\n"
        "Usage: lattice-char-index-utterance [options] separator-symbols lat-rspecifier index-wspecifier\n"
        " e.g.: lattice-char-index-utterance \"3 4\" ark:1.lats ark:1.index\n";
#elif KLU_TOOL == 3 /* KLU_FRAME_POST */
    const char* usage =
        "Compute the posterior log-probability of each word for each given utterance frame. That is, we compute "
        "log P(a_i = v | x), for all possible utterance frames i and words v.\n\n"
        "Usage: lattice-to-word-frame-post [options] lat-rspecifier post-wspecifier\n"
        " e.g.: lattice-to-word-frame-post --acoustic-scale=0.1 ark:1.lats ark:1.word.pos.post\n";
#elif KLU_TOOL == 10 /* KLU_LENGTH_DIST */
    const char* usage =
        "Compute the distribution of the length of the transcriptions in a lattice.\n\n"
        "Usage: lattice-to-transcript-length-dist [options] lattice-rspecifier1 posterior-wspecifier\n"
        " e.g.: lattice-to-transcript-length-dist ark:1.lats ark:1.posts\n";
#elif KLU_TOOL == 8 /* KLU_POSITION_POST */
    const char* usage =
        "Compute the posterior log-probability of each word for each given transcription position. That is, we "
        "compute log P(w_k = v | x), for all possible transcript position k, and words v.\n\n"
        "Usage: lattice-to-word-position-post [options] lat-rspecifier post-wspecifier [segm-wspecifier]\n"
        " e.g.: lattice-to-word-position-post --acoustic-scale=0.1 ark:1.lats ark:1.word.pos.post\n"
        "See also: lattice-to-word-frame-post\n";
#elif KLU_TOOL == 4 /* KLU_PRUNE_DYN_BEAM */
    const char* usage =
        "Iteratively reduce the beam of the lattice until a maximum number of arcs and states is achieved.\n\n"
        "Usage: lattice-prune-dyn-beam [options] lat-rspecifier lat-wspecifier\n";
#elif KLU_TOOL == 11 /* KLU_PRUNE_ARCS */
    const char* usage =
        "Iteratively reduce the beam of the lattice until a maximum number of arcs and states is achieved.\n\n"
        "Usage: lattice-prune-arcs [options] lat-rspecifier lat-wspecifier\n";  // (the reference's own text)
#elif KLU_TOOL == 5 /* KLU_BEST_PATH2 */
    const char* usage =
        "Generate especial 1-best path through lattices, which minimizes the expected number of position-wise "
        "errors (an upper bound of the expected Levenshtein distance) instead of the 0-1 sequence loss.\n\n"
        "Usage: lattice-best-path2 [options] lat-rspecifier [transcriptions-wspecifier]\n";
#endif
    ParseOptions po(usage);
    po.Register("acoustic-scale", &acoustic_scale, "Scaling factor for acoustic likelihoods in the lattices.");
    po.Register("graph-scale", &graph_scale, "Scaling factor for graph probabilities in the lattices.");
    po.Register("insertion-penalty", &insertion_penalty,
                "Add this penalty to the lattice arcs with non-epsilon output label (typically, equivalent to word "
                "insertion penalty).");
#if KLU_TOOL == 1 /* KLU_POSITION */ || KLU_TOOL == 0 /* KLU_SEGMENT */ || KLU_TOOL == 2 /* KLU_UTTERANCE */ || KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
    po.Register("beam", &beam, "Pruning beam (applied after acoustic scaling and adding the insertion penalty).");
    po.Register("num-threads", &num_threads, "Accepted for compatibility; lattices are batched on the GPU instead.");
    po.Register("num-threads-total", &num_threads_total, "Accepted for compatibility; ignored.");
#endif
#if KLU_TOOL == 1 /* KLU_POSITION */ || KLU_TOOL == 0 /* KLU_SEGMENT */ || KLU_TOOL == 2 /* KLU_UTTERANCE */
    po.Register("exclude-words", &exclude_str,
                "Space-separated list of integers representing the words to exclude from the index.");
    po.Register("include-words", &include_str,
                "Space-separated list of integers representing the words to include in the index.");
#endif
#if KLU_TOOL == 2 /* KLU_UTTERANCE */
    int32_t rho_label = INT_MAX;
    po.Register("rho-label", &rho_label, "Accepted for compatibility (no composition is materialised).");
#endif
#if KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
    float determinize_delta = 1.0f / 1024.0f / 8.0f;
    po.Register("nbest", &st.opts.nbest, "Extract this number of n-best hypothesis.");
    po.Register("determinize-delta", &determinize_delta,
                "Accepted for compatibility (sums are exact here, no determinization quantisation).");
    po.Register("other-groups", &other_groups_str,
                "Specific labels to group as words. Groups are separated with a semicolon, labels within a group "
                "with spaces.");
#endif
#if KLU_TOOL == 11 /* KLU_PRUNE_ARCS */
    po.Register("beam", &beam, "");  // latbin/lattice-prune-arcs.cc:117
#endif
#if KLU_TOOL == 4 /* KLU_PRUNE_DYN_BEAM */
    po.Register("beam-ratio", &st.opts.beam_ratio, "Reduce the maximum beam by this ratio at each iteration.");
    po.Register("min-beam", &st.opts.min_beam, "Minimum beam threshold");
    po.Register("max-arcs", &st.opts.max_arcs, "Maximum number of arcs of each lattice.");
    po.Register("max-states", &st.opts.max_states, "Maximum number of states of each lattice.");
#endif
    po.Read(argc, argv);

#if KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
    if (po.NumArgs() != 3) {
      po.PrintUsage();
      exit(1);
    }
    const int kLatArg = 2;
#elif KLU_TOOL == 8 /* KLU_POSITION_POST */
    if (po.NumArgs() != 2 && po.NumArgs() != 3) {  // latbin/lattice-to-word-position-post.cc:60-63
      po.PrintUsage();
      exit(1);
    }
    const int kLatArg = 1;
#elif KLU_TOOL == 5 /* KLU_BEST_PATH2 */
    if (po.NumArgs() < 1 || po.NumArgs() > 2) {
      po.PrintUsage();
      exit(1);
    }
    const int kLatArg = 1;
#elif KLU_TOOL == 4 /* KLU_PRUNE_DYN_BEAM */
    if (po.NumArgs() < 2) {
      po.PrintUsage();
      exit(1);
    }
    const int kLatArg = 1;
    if (st.opts.beam_ratio <= 0.0 || st.opts.beam_ratio >= 1.0)
      KIO_ERR("--beam_ratio must be in the open range (0.0, 1.0).");
#elif KLU_TOOL == 11 /* KLU_PRUNE_ARCS */
    if (po.NumArgs() < 2) {
      po.PrintUsage();
      exit(1);
    }
    const int kLatArg = 1;
    if (beam <= 0.0) KIO_ERR("--beam_ratio must be in the open range (0.0, inf).");  // :131-133 (sic)
#else
    if (po.NumArgs() != 2) {
      po.PrintUsage();
      exit(1);
    }
    const int kLatArg = 1;
#endif
    st.opts.acoustic_scale = acoustic_scale;
    st.opts.graph_scale = graph_scale;
    st.opts.insertion_penalty = insertion_penalty;
    st.opts.beam = beam;
    if (!SplitStringToIntegers(exclude_str, " ", true, &st.exclude)) KIO_ERR("Invalid --exclude-words");
    if (!SplitStringToIntegers(include_str, " ", true, &st.include)) KIO_ERR("Invalid --include-words");
    {
      std::set<int32_t> a(st.exclude.begin(), st.exclude.end()), b(st.include.begin(), st.include.end());
      st.exclude.assign(a.begin(), a.end());
      st.include.assign(b.begin(), b.end());
    }
    st.opts.include_words = st.include.data();
    st.opts.num_include = (int32_t)st.include.size();
    st.opts.exclude_words = st.exclude.data();
    st.opts.num_exclude = (int32_t)st.exclude.size();
#if KLU_TOOL == 6 /* KLU_CHAR_POSITION */ || KLU_TOOL == 9 /* KLU_CHAR_SEGMENT */ || KLU_TOOL == 12 /* KLU_CHAR_UTTERANCE */
    {
      // kwsbin2/utils.h:41-84 ParseSeparatorGroups
      std::map<int32_t, int32_t> label_group;
      label_group[0] = 0;
      st.inc_groups.push_back(INT_MAX);
      std::vector<int32_t> ws;
      if (!SplitStringToIntegers(po.GetArg(1), " ", true, &ws)) KIO_ERR("Invalid whitespace label list");
      if (ws.empty()) KIO_ERR("At least one label must be specified as a whitespace separator!");
      auto assign = [&](int32_t group, const std::vector<int32_t>& labels) {
        for (int32_t lab : labels) {
          auto r = label_group.emplace(lab, group);
          if (!r.second)
            KIO_ERR("Each label must be assigned to one group at most. Label " << lab << " was assigned to both groups "
                                                                               << r.first->second << " and " << group << ".");
        }
      };
      assign(1, ws);
      size_t start = 0;
      int32_t gi = 0;
      while (start <= other_groups_str.size()) {
        size_t end = other_groups_str.find(';', start);
        if (end == std::string::npos) end = other_groups_str.size();
        const std::string grp = other_groups_str.substr(start, end - start);
        if (grp.find_first_not_of(" \t") != std::string::npos) {
          std::vector<int32_t> labs;
          if (!SplitStringToIntegers(grp, " ", true, &labs)) KIO_ERR("Invalid --other-groups");
          assign(gi + 2, labs);
          st.inc_groups.push_back(gi + 2);
          ++gi;
        }
        start = end + 1;
      }
      for (auto& kv : label_group) {
        st.group_labels.push_back(kv.first);
        st.group_ids.push_back(kv.second);
      }
      st.del_groups.push_back(1);
      st.opts.group_labels = st.group_labels.data();
      st.opts.group_ids = st.group_ids.data();
      st.opts.num_group_labels = (int32_t)st.group_labels.size();
      st.opts.inc_groups = st.inc_groups.data();
      st.opts.num_inc_groups = (int32_t)st.inc_groups.size();
      st.opts.del_groups = st.del_groups.data();
      st.opts.num_del_groups = (int32_t)st.del_groups.size();
    }
#endif
    // KLU_DEVICES=0,1,... : one context (stream, buffers) per listed GPU; KLU_DEVICE=n for one
    {
      std::vector<int32_t> devs;
      if (const char* e = getenv("KLU_DEVICES")) {
        std::string str(e);
        for (char& ch : str)
          if (ch == ',') ch = ' ';
        if (!SplitStringToIntegers(str, " ", true, &devs) || devs.empty()) KIO_ERR("Invalid KLU_DEVICES");
      } else {
        const char* dev_env = getenv("KLU_DEVICE");
        devs.push_back(dev_env ? atoi(dev_env) : 0);
      }
      for (int32_t d : devs) {
        klu_ctx* ctx = nullptr;
        KLU_CHECK(klu_create(d, &ctx));
        st.ctxs.push_back(ctx);
      }
    }
    int64_t batch_arcs = (int64_t)32 << 20;
    if (const char* e = getenv("KLU_BATCH_ARCS")) batch_arcs = std::max<long long>(1, atoll(e));

    const std::string lattice_rspecifier = po.GetArg(kLatArg);
    TableWriter writer(po.GetOptArg(kLatArg + 1));
    st.writer = &writer;
    const bool keep = KLU_TOOL == 4 /* KLU_PRUNE_DYN_BEAM */ || KLU_TOOL == 11 /* KLU_PRUNE_ARCS */;
    {
      Pipeline pipe(&st);
      Batch batch;
      bool ok = true;
      auto t_read = std::chrono::steady_clock::now();
      SequentialCompactLatticeReader reader(lattice_rspecifier, keep);
      std::vector<CompactLat> block;
      while (ok && !reader.Done()) {
        if (reader.ReadBlock(batch_arcs - batch.arcs(), &block, kMaxBatchLattices - batch.lats.size())) {
          batch.AddBlock(&block, keep);  // in-memory archive: parsed in parallel
        } else {
          batch.Add(std::move(reader.Value()), keep);
          reader.Next();
        }
        if (batch.arcs() >= batch_arcs || batch.lats.size() >= kMaxBatchLattices) {
          const auto t1 = std::chrono::steady_clock::now();
          st.sec_read += std::chrono::duration<double>(t1 - t_read).count();
          ok = pipe.Submit(std::move(batch));
          batch = Batch();
          t_read = std::chrono::steady_clock::now();
          st.sec_wait += std::chrono::duration<double>(t_read - t1).count();
        }
      }
      st.sec_read += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_read).count();
      if (ok && !batch.lats.empty()) pipe.Submit(std::move(batch));
      pipe.Finish();
    }
    if (writer.IsOpen()) writer.Close();
    if (getenv("KLU_TRACE"))
      KIO_LOG("time: reading " << st.sec_read << " s, waiting for the pipeline " << st.sec_wait << " s, GPU calls " << st.sec_gpu
                             << " s, writing " << st.sec_emit << " s");
#if KLU_TOOL == 5 /* KLU_BEST_PATH2 */
    KIO_LOG("Overall cost per frame is " << (st.total_cost / st.total_frames) << " over " << st.total_frames
                                         << " frames.");
#endif
    for (klu_ctx* ctx : st.ctxs) klu_destroy(ctx);
    return 0;
  } catch (const std::exception& e) {
    std::cerr << e.what();
    return kErrorCode;
  }
}
