// CPU reference of lattice-char-index-utterance: test infrastructure like oracle/klu_oracle.cc, whose
// lattice reader, prologue, label-group split and result table it reuses by inclusion.  The tests
// compile it into a temporary directory (tests/char_utterance_ref.py).
#include "../oracle/klu_oracle.cc"

// lattice-char-index-utterance (no reference binary; DESIGN.md section 7).  The prologue,
// label groups and runs are those of CharIndexPosition without the word-count split; a
// pseudo-word v's value is log P(some run of the path spells v) - total, a probability (a
// path with two runs spelling v counts once).  The strings come from the same run search
// as CharIndexPosition; each value from a first-occurrence DP over the split lattice:
//   a0[s]    mass of the paths start -> s that are not inside a run matching a prefix of v
//            and have completed no occurrence of v;
//   a[s][j]  the same, inside a run of v's group whose labels so far spell v[0..j).
// An arc that leaves a run (group change) after j = |v| completes an occurrence, as does a
// final weight; completed mass goes to the result with the whole rest of the path (bw).
// Rows: the nbest best by (logp desc, string asc).
double CharOccurrenceLogSum(const SplitLat& sp, const std::vector<int32>& order, const std::vector<double>& bw,
                            const std::vector<int32>& v, int32 gv) {
  const Lat& lat = sp.lat;
  const int32 n = lat.NumStates(), m = (int32)v.size();
  std::vector<double> a0(n, kLogZeroDouble), a((size_t)n * (m + 1), kLogZeroDouble);
  a0[0] = 0.0;
  double res = kLogZeroDouble;
  for (int32 s : order) {
    const double* as = &a[(size_t)s * (m + 1)];
    if (as[m] != kLogZeroDouble && lat.IsFinal(s)) res = LogAdd(res, as[m] - Cost(lat.fg[s], lat.fa[s]));
    for (const auto& arc : lat.out[s]) {
      const int32 y = arc.next, gy = sp.group[y];
      const double w = -Cost(arc.g, arc.a);
      const bool newrun = s == 0 || sp.group[s] != gy;
      double* ay = &a[(size_t)y * (m + 1)];
      if (a0[s] != kLogZeroDouble) {
        if (newrun && gy == gv && arc.label == v[0]) ay[1] = LogAdd(ay[1], a0[s] + w);
        else a0[y] = LogAdd(a0[y], a0[s] + w);
      }
      for (int32 j = 1; j <= m; ++j) {
        if (as[j] == kLogZeroDouble) continue;
        if (newrun) {
          if (j == m) res = LogAdd(res, as[j] + w + bw[y]);
          else a0[y] = LogAdd(a0[y], as[j] + w);
        } else if (j < m && arc.label == v[j]) {
          ay[j + 1] = LogAdd(ay[j + 1], as[j] + w);
        } else {
          a0[y] = LogAdd(a0[y], as[j] + w);  // a run longer than v, or another string
        }
      }
    }
  }
  return res;
}

struct CharUttRow {
  std::string s;
  double logp;
};

void EmitCharUtterance(std::vector<CharUttRow>* rows, const Opts& o, double total, Result* r) {
  std::sort(rows->begin(), rows->end(), [](const CharUttRow& a, const CharUttRow& b) {
    if (a.logp != b.logp) return a.logp > b.logp;
    return a.s < b.s;
  });
  if ((int64_t)rows->size() > (int64_t)o.nbest) rows->resize(std::max<int32>(o.nbest, 0));
  for (const auto& row : *rows) {
    r->str.push_back(row.s);
    r->d0.push_back(row.logp);
  }
  r->ds0 = total;
}

std::string JoinLabels(const std::vector<int32>& chars) {
  std::string s;
  for (size_t i = 0; i < chars.size(); ++i) {
    if (i) s += "_";
    s += std::to_string(chars[i]);
  }
  return s;
}

void CharIndexUtterance(Lat lat0, const Opts& o0, Result* r) {
  Opts o = o0;
  o.group_inc.clear();  // strings only: every split state has count 0
  Prologue(&lat0, o, true);
  if (lat0.Empty()) return;
  SplitLat sp;
  SplitByGroupAndCount(lat0, o, &sp);
  const Lat& lat = sp.lat;
  const int32 n = lat.NumStates();
  std::vector<int32> indeg(n, 0), order;
  for (int32 s = 0; s < n; ++s)
    for (const auto& arc : lat.out[s]) indeg[arc.next]++;
  {
    std::vector<int32> st;
    for (int32 s = n - 1; s >= 0; --s)
      if (indeg[s] == 0) st.push_back(s);
    while (!st.empty()) {
      int32 s = st.back();
      st.pop_back();
      order.push_back(s);
      for (const auto& arc : lat.out[s])
        if (--indeg[arc.next] == 0) st.push_back(arc.next);
    }
  }
  std::vector<double> bw(n, kLogZeroDouble);
  for (auto it = order.rbegin(); it != order.rend(); ++it) {
    const int32 s = *it;
    double b = -Cost(lat.fg[s], lat.fa[s]);
    for (const auto& arc : lat.out[s]) b = LogAdd(b, bw[arc.next] - Cost(arc.g, arc.a));
    bw[s] = b;
  }
  const double total = bw[0];
  std::vector<double> exitw(n, kLogZeroDouble);
  for (int32 u = 0; u < n; ++u) {
    double e = -Cost(lat.fg[u], lat.fa[u]);
    for (const auto& arc : lat.out[u])
      if (sp.group[arc.next] != sp.group[u]) e = LogAdd(e, -Cost(arc.g, arc.a) + bw[arc.next]);
    exitw[u] = e;
  }
  // the run search of CharIndexPosition: every string some run spells (and can end with), with
  // the log-sum of its runs, log E[N(v)] + total (N(v) = runs of the path that spell v)
  std::map<std::vector<int32>, std::pair<int32, double> > strings;  // chars -> (group, runs' mass)
  auto visit = [&](const std::vector<int32>& chars, int32 g, int32 x, double w) {
    if (exitw[x] == kLogZeroDouble) return;
    auto it = strings.emplace(chars, std::make_pair(g, kLogZeroDouble)).first;
    it->second.second = LogAdd(it->second.second, w + exitw[x]);
  };
  std::vector<double> fw(n, kLogZeroDouble);
  fw[0] = 0.0;
  for (int32 s : order)
    for (const auto& arc : lat.out[s]) fw[arc.next] = LogAdd(fw[arc.next], fw[s] - Cost(arc.g, arc.a));
  struct Frame { int32 state; size_t arc; };
  for (int32 u = 0; u < n; ++u) {
    for (const auto& first : lat.out[u]) {
      const int32 v1 = first.next;
      if (!(u == 0 || sp.group[u] != sp.group[v1])) continue;
      const int32 g = sp.group[v1];
      if (o.delete_groups.count(g) || g == 0) continue;
      std::vector<int32> chars(1, first.label);
      std::vector<Frame> stack(1, Frame{v1, 0});
      std::vector<double> wstack(1, fw[u] - Cost(first.g, first.a));
      visit(chars, g, v1, wstack.back());
      while (!stack.empty()) {
        Frame& f = stack.back();
        if (f.arc >= lat.out[f.state].size()) {
          stack.pop_back();
          wstack.pop_back();
          if (!stack.empty()) chars.pop_back();
          continue;
        }
        const Arc& arc = lat.out[f.state][f.arc++];
        if (sp.group[arc.next] != g || f.state == 0) continue;
        chars.push_back(arc.label);
        stack.push_back(Frame{arc.next, 0});
        wstack.push_back(wstack.back() - Cost(arc.g, arc.a));
        visit(chars, g, arc.next, wstack.back());
      }
    }
  }
  // P(v) <= E[N(v)]: the DP runs in decreasing E order and stops once E is below the nbest-th
  // best P found (tau); strings left out cannot reach the rows, ties at tau included
  std::vector<std::pair<double, const std::vector<int32>*> > byE;
  for (const auto& kv : strings) byE.push_back(std::make_pair(kv.second.second, &kv.first));
  std::stable_sort(byE.begin(), byE.end(), [](const std::pair<double, const std::vector<int32>*>& a,
                                              const std::pair<double, const std::vector<int32>*>& b) { return a.first > b.first; });
  std::vector<CharUttRow> rows;
  std::priority_queue<double, std::vector<double>, std::greater<double> > best;  // the nbest best values
  for (const auto& e : byE) {
    if (o.nbest <= 0) break;
    if ((int32)best.size() >= o.nbest && e.first - total < best.top() - 1e-9 * (1.0 + std::fabs(best.top()))) break;
    const double lp = CharOccurrenceLogSum(sp, order, bw, *e.second, strings[*e.second].first) - total;
    rows.push_back(CharUttRow{JoinLabels(*e.second), lp});
    best.push(lp);
    if ((int32)best.size() > o.nbest) best.pop();
  }
  EmitCharUtterance(&rows, o, total, r);
}

// The same rows by their definition: every complete path of a (tiny) lattice is cut into
// maximal runs of one label group; each string that a run outside groups 0 and the deleted
// groups spells gets the path's weight once.
void BruteCharUtterance(Lat lat, const Opts& o, Result* r) {
  Prologue(&lat, o, true);
  if (lat.Empty()) return;
  std::map<std::string, double> acc;
  double total = kLogZeroDouble;
  std::vector<const Arc*> path;
  std::function<void(int32, double)> rec = [&](int32 s, double w) {
    if (lat.IsFinal(s)) {
      const double pw = w - Cost(lat.fg[s], lat.fa[s]);
      total = LogAdd(total, pw);
      std::set<std::string> seen;
      for (size_t i = 0; i < path.size();) {
        const int32 g = GroupOf(path[i]->label, o);
        std::vector<int32> chars;
        size_t k = i;
        for (; k < path.size() && GroupOf(path[k]->label, o) == g; ++k) chars.push_back(path[k]->label);
        if (g != 0 && !o.delete_groups.count(g)) seen.insert(JoinLabels(chars));
        i = k;
      }
      for (const auto& str : seen) {
        auto it = acc.find(str);
        if (it == acc.end()) acc.emplace(str, pw);
        else it->second = LogAdd(it->second, pw);
      }
    }
    for (const auto& arc : lat.out[s]) {
      path.push_back(&arc);
      rec(arc.next, w - Cost(arc.g, arc.a));
      path.pop_back();
    }
  };
  rec(0, 0.0);
  std::vector<CharUttRow> rows;
  for (const auto& kv : acc) rows.push_back(CharUttRow{kv.first, kv.second - total});
  EmitCharUtterance(&rows, o, total, r);
}


extern "C" {

enum { REF_CHAR_UTTERANCE = 0, REF_BRUTE_CHAR_UTTERANCE = 1 };

void* charutt_run(int tool, const ora_lat* l, const ora_opts* o) {
  Result* r = new Result();
  const Opts opts = ConvertOpts(o);
  Lat lat = BuildLat(l->nstates, l->narcs, l->src, l->dst, l->label, l->dur, l->graph, l->acoustic, l->fin_graph,
                     l->fin_acoustic, l->fin_dur, &r->error, false);
  if (!r->error.empty()) return r;
  if (tool == REF_CHAR_UTTERANCE) CharIndexUtterance(lat, opts, r);
  else if (tool == REF_BRUTE_CHAR_UTTERANCE) BruteCharUtterance(lat, opts, r);
  else r->error = "unknown tool";
  return r;
}

}  // extern "C"
