"""ctypes binding of include/klu.h (libklu_b200.so).

This is plumbing for tests and bench.py; the reference-facing host code is the
C++ tools under host/.  There is no CPU fallback: Engine() raises when the CUDA
library is missing or no GPU is usable.
"""
import ctypes as C
import json
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

SEGMENT, POSITION, UTTERANCE, FRAME_POST, PRUNE_DYN_BEAM, BEST_PATH2, CHAR_POSITION, FWD_BWD, POSITION_POST, CHAR_SEGMENT, LENGTH_DIST, PRUNE_ARCS, CHAR_UTTERANCE = range(13)
TOOL_NAMES = {SEGMENT: "lattice-word-index-segment", POSITION: "lattice-word-index-position",
              UTTERANCE: "lattice-word-index-utterance", FRAME_POST: "lattice-to-word-frame-post",
              PRUNE_DYN_BEAM: "lattice-prune-dyn-beam", BEST_PATH2: "lattice-best-path2",
              CHAR_POSITION: "lattice-char-index-position", FWD_BWD: "fwd-bwd",
              POSITION_POST: "lattice-to-word-position-post", CHAR_SEGMENT: "lattice-char-index-segment",
              LENGTH_DIST: "lattice-to-transcript-length-dist", PRUNE_ARCS: "lattice-prune-arcs",
              CHAR_UTTERANCE: "lattice-char-index-utterance"}
INT_MAX = 2**31 - 1

# every symbol include/klu.h declares (checked by tests/test_capi_symbols.py)
SYMBOLS = ["klu_last_error", "klu_version", "klu_opts_default", "klu_device_count", "klu_create", "klu_destroy",
           "klu_host_alloc", "klu_host_free", "klu_topsort", "klu_load", "klu_run", "klu_sync", "klu_result_offsets",
           "klu_fetch_segment", "klu_fetch_position", "klu_fetch_utterance", "klu_fetch_frame_post", "klu_fetch_frame_post_csr", "klu_fetch_position_post", "klu_fetch_length_dist",
           "klu_fetch_best_path2", "klu_fetch_prune", "klu_result_char_sizes", "klu_fetch_char_position", "klu_fetch_char_segment",
           "klu_fetch_char_utterance",
           "klu_fetch_fwd_bwd", "klu_timer_start", "klu_timer_stop", "klu_launch_count", "klu_profile_enable",
           "klu_profile_json", "klu_batch_stats", "klu_flush_l2", "klu_load_times"]


class KluLattices(C.Structure):
    _fields_ = [("num_lattices", C.c_int32), ("state_off", C.c_void_p), ("arc_off", C.c_void_p),
                ("arc_src", C.c_void_p), ("arc_dst", C.c_void_p), ("arc_label", C.c_void_p), ("arc_dur", C.c_void_p),
                ("arc_graph", C.c_void_p), ("arc_acoustic", C.c_void_p), ("fin_graph", C.c_void_p),
                ("fin_acoustic", C.c_void_p), ("fin_dur", C.c_void_p), ("state_num_arcs", C.c_void_p),
                ("arc_dur_u8", C.c_void_p), ("arc_dst_delta_u16", C.c_void_p), ("arc_label_u16", C.c_void_p)]


class KluOpts(C.Structure):
    _fields_ = [("acoustic_scale", C.c_float), ("graph_scale", C.c_float), ("insertion_penalty", C.c_float),
                ("beam", C.c_float), ("include_words", C.c_void_p), ("num_include", C.c_int32),
                ("exclude_words", C.c_void_p), ("num_exclude", C.c_int32), ("beam_ratio", C.c_float),
                ("min_beam", C.c_float), ("max_arcs", C.c_int32), ("max_states", C.c_int32), ("nbest", C.c_int32),
                ("group_labels", C.c_void_p), ("group_ids", C.c_void_p), ("num_group_labels", C.c_int32),
                ("inc_groups", C.c_void_p), ("num_inc_groups", C.c_int32), ("del_groups", C.c_void_p),
                ("num_del_groups", C.c_int32)]


_LIB = None


def lib_path():
    return os.path.join(_HERE, "libklu_b200.so")


def lib():
    global _LIB
    if _LIB is None:
        p = lib_path()
        if not os.path.exists(p):
            raise RuntimeError("%s is not built (run __graft_entry__.build()); there is no CPU fallback" % p)
        L = C.CDLL(p)
        L.klu_last_error.restype = C.c_char_p
        for name in SYMBOLS:
            getattr(L, name)  # fail loudly on a missing export
        _LIB = L
    return _LIB


class KluError(RuntimeError):
    pass


def _chk(rc):
    if rc != 0:
        raise KluError(lib().klu_last_error().decode())


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None and a.size else None


def _i32(v):
    return np.ascontiguousarray(np.asarray(list(v), dtype=np.int32))


def char_groups(wspace, other_groups=()):
    """kwsbin2/utils.h:41-84 ParseSeparatorGroups."""
    label_group = {0: 0}
    for w in wspace:
        if w in label_group:
            raise ValueError("label %d assigned to two groups" % w)
        label_group[w] = 1
    inc = [INT_MAX]
    for gi, grp in enumerate(other_groups):
        for lab in grp:
            if lab in label_group:
                raise ValueError("label %d assigned to two groups" % lab)
            label_group[lab] = gi + 2
        inc.append(gi + 2)
    return label_group, inc, [1]


def compact_arcs(batch):
    """(dur_u8, dst_delta_u16) of a batch -- klu_lattices.arc_dur_u8 / arc_dst_delta_u16 -- or None
    for a form that does not fit (a duration over 255, a destination more than 65535 states ahead)."""
    dur8 = batch.dur.astype(np.uint8) if batch.dur.size == 0 or (batch.dur.min() >= 0 and batch.dur.max() < 256) else None
    delta = batch.dst - batch.src
    d16 = delta.astype(np.uint16) if delta.size == 0 or (delta.min() >= 0 and delta.max() < 65536) else None
    return dur8, d16


def compact_labels(batch):
    """klu_lattices.arc_label_u16 of a batch, or None when a label does not fit 16 bits."""
    lab = batch.label
    return lab.astype(np.uint16) if lab.size == 0 or (lab.min() >= 0 and lab.max() < 65536) else None


def make_opts(acoustic_scale=1.0, graph_scale=1.0, insertion_penalty=0.0, beam=float("inf"), include_words=(),
              exclude_words=(), beam_ratio=0.9, min_beam=1e-3, max_arcs=INT_MAX, max_states=INT_MAX, nbest=100,
              label_group=None, inc_groups=(), del_groups=()):
    o = KluOpts()
    lib().klu_opts_default(C.byref(o))
    keep = [_i32(include_words), _i32(exclude_words)]
    lg = label_group or {}
    keep += [_i32(lg.keys()), _i32(lg.values()), _i32(inc_groups), _i32(del_groups)]
    o.acoustic_scale, o.graph_scale, o.insertion_penalty, o.beam = acoustic_scale, graph_scale, insertion_penalty, beam
    o.include_words, o.num_include = _p(keep[0]), keep[0].size
    o.exclude_words, o.num_exclude = _p(keep[1]), keep[1].size
    o.beam_ratio, o.min_beam, o.max_arcs, o.max_states, o.nbest = beam_ratio, min_beam, max_arcs, max_states, nbest
    o.group_labels, o.group_ids, o.num_group_labels = _p(keep[2]), _p(keep[3]), keep[2].size
    o.inc_groups, o.num_inc_groups = _p(keep[4]), keep[4].size
    o.del_groups, o.num_del_groups = _p(keep[5]), keep[5].size
    return o, keep


class Engine:
    """One context on one GPU (klu_create .. klu_destroy)."""

    def __init__(self, device=0):
        self.L = lib()
        self.h = C.c_void_p()
        _chk(self.L.klu_create(device, C.byref(self.h)))
        self.batch = None
        self._keep = None

    def close(self):
        if self.h:
            self.L.klu_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- memory ---------------------------------------------------------------
    def pinned(self, nbytes):
        """Pinned host buffer (klu_host_alloc) as a writable memoryview-able object."""
        p = C.c_void_p()
        _chk(self.L.klu_host_alloc(C.c_size_t(nbytes), C.byref(p)))
        buf = (C.c_char * nbytes).from_address(p.value)
        return buf

    # -- data -----------------------------------------------------------------
    def load(self, batch, state_num_arcs=None, dur_u8=None, dst_delta_u16=None, label_u16=None):
        """state_num_arcs (optional, int32 per state): upload without the per-arc source array;
        dur_u8 / dst_delta_u16 / label_u16 (optional, see compact_arcs(), compact_labels()): the compact
        forms of arc_dur / arc_dst / arc_label."""
        kl = KluLattices(len(batch), _p(batch.state_off), _p(batch.arc_off),
                         None if state_num_arcs is not None else _p(batch.src),
                         None if dst_delta_u16 is not None else _p(batch.dst),
                         None if label_u16 is not None else _p(batch.label),
                         None if dur_u8 is not None else _p(batch.dur), _p(batch.graph),
                         _p(batch.acoustic), _p(batch.fin_graph),
                         _p(batch.fin_acoustic), _p(batch.fin_dur), _p(state_num_arcs), _p(dur_u8), _p(dst_delta_u16),
                         _p(label_u16))
        _chk(self.L.klu_load(self.h, C.byref(kl)))
        self.batch = batch

    def run(self, tool, **opts):
        o, keep = make_opts(**opts)
        _chk(self.L.klu_run(self.h, tool, C.byref(o)))

    def run_opts(self, tool, o):
        _chk(self.L.klu_run(self.h, tool, C.byref(o)))

    def sync(self):
        _chk(self.L.klu_sync(self.h))

    # -- results --------------------------------------------------------------
    def offsets(self):
        off = np.zeros(len(self.batch) + 1, np.int64)
        _chk(self.L.klu_result_offsets(self.h, _p(off)))
        return off

    def fetch_segment(self):
        off = self.offsets()
        n = int(off[-1])
        w, t0, t1 = (np.zeros(n, np.int32) for _ in range(3))
        lp = np.zeros(n, np.float64)
        _chk(self.L.klu_fetch_segment(self.h, _p(w), _p(t0), _p(t1), _p(lp)))
        return off, w, t0, t1, lp

    def fetch_position(self):
        off = self.offsets()
        n = int(off[-1])
        w, pos, t0, t1 = (np.zeros(n, np.int32) for _ in range(4))
        lp = np.zeros(n, np.float64)
        _chk(self.L.klu_fetch_position(self.h, _p(w), _p(pos), _p(t0), _p(t1), _p(lp)))
        return off, w, pos, t0, t1, lp

    def fetch_utterance(self):
        off = self.offsets()
        n = int(off[-1])
        w = np.zeros(n, np.int32)
        lp = np.zeros(n, np.float64)
        _chk(self.L.klu_fetch_utterance(self.h, _p(w), _p(lp)))
        return off, w, lp

    def pinned_array(self, dtype, count):
        """numpy array backed by pinned host memory (klu_host_alloc)."""
        buf = self.pinned(max(int(count), 1) * np.dtype(dtype).itemsize)
        self._pinned_keep = getattr(self, "_pinned_keep", [])
        self._pinned_keep.append(buf)
        return np.frombuffer(buf, dtype=dtype, count=int(count))

    def fetch_frame_post(self, out=None):
        """out: optional (frame, word, logp) arrays (e.g. pinned) of sufficient size."""
        off = self.offsets()
        n = int(off[-1])
        nf = np.zeros(len(self.batch), np.int32)
        if out is not None and out[0].size >= n:
            fr, w, lp = out[0][:n], out[1][:n], out[2][:n]
        else:
            fr, w = np.zeros(n, np.int32), np.zeros(n, np.int32)
            lp = np.zeros(n, np.float32)
        _chk(self.L.klu_fetch_frame_post(self.h, _p(nf), _p(fr), _p(w), _p(lp)))
        return off, nf, fr, w, lp

    def fetch_frame_post_csr(self, out=None):
        """Rows without the per-row frame column: (off, num_frames, frame_row_off, word, logp); lattice l's
        frame_row_off entries start at sum(num_frames[:l] + 1).  out: optional (frame_row_off, word, logp)
        arrays (e.g. pinned) of sufficient size."""
        off = self.offsets()
        n = int(off[-1])
        nf = np.zeros(len(self.batch), np.int32)
        _chk(self.L.klu_fetch_frame_post_csr(self.h, _p(nf), None, None, None))  # frame counts only: sizes frame_row_off
        slots = int(nf.sum(dtype=np.int64)) + len(nf)
        if out is not None and out[0].size >= slots and out[1].size >= n:
            fo, w, lp = out[0][:slots], out[1][:n], out[2][:n]
        else:
            fo, w, lp = np.zeros(slots, np.int64), np.zeros(n, np.int32), np.zeros(n, np.float32)
        _chk(self.L.klu_fetch_frame_post_csr(self.h, _p(nf), _p(fo), _p(w), _p(lp)))
        return off, nf, fo, w, lp

    def fetch_position_post(self):
        off = self.offsets()
        n = int(off[-1])
        npos = np.zeros(len(self.batch), np.int32)
        pos, w = np.zeros(n, np.int32), np.zeros(n, np.int32)
        lp = np.zeros(n, np.float32)
        _chk(self.L.klu_fetch_position_post(self.h, _p(npos), _p(pos), _p(w), _p(lp)))
        return off, npos, pos, w, lp

    def fetch_best_path2(self):
        off = self.offsets()
        n = int(off[-1])
        lab = np.zeros(n, np.int32)
        cost = np.zeros(len(self.batch), np.float32)
        nf = np.zeros(len(self.batch), np.int32)
        _chk(self.L.klu_fetch_best_path2(self.h, _p(lab), _p(cost), _p(nf)))
        return off, lab, cost, nf

    def fetch_prune(self):
        off = self.offsets()
        n = int(off[-1])
        b = self.batch
        ai, ns, nd = (np.zeros(n, np.int32) for _ in range(3))
        g, a = np.zeros(n, np.float32), np.zeros(n, np.float32)
        smap = np.zeros(b.num_states, np.int32)
        fg, fa = np.zeros(b.num_states, np.float32), np.zeros(b.num_states, np.float32)
        beams = np.zeros(2 * len(b), np.float64)
        _chk(self.L.klu_fetch_prune(self.h, _p(ai), _p(ns), _p(nd), _p(g), _p(a), _p(smap), _p(fg), _p(fa),
                                    _p(beams)))
        return off, ai, ns, nd, g, a, smap, fg, fa, beams

    def fetch_char_position(self):
        off = self.offsets()
        n = int(off[-1])
        tot = C.c_int64()
        _chk(self.L.klu_result_char_sizes(self.h, C.byref(tot)))
        coff = np.zeros(n + 1, np.int64)
        chars = np.zeros(tot.value, np.int32)
        pos, t0, t1 = (np.zeros(n, np.int32) for _ in range(3))
        lp = np.zeros(n, np.float64)
        _chk(self.L.klu_fetch_char_position(self.h, _p(coff), _p(chars), _p(pos), _p(t0), _p(t1), _p(lp)))
        return off, coff, chars, pos, t0, t1, lp

    def fetch_fwd_bwd(self):
        b = self.batch
        al, be = np.zeros(b.num_states, np.float64), np.zeros(b.num_states, np.float64)
        tot = np.zeros(len(b), np.float64)
        _chk(self.L.klu_fetch_fwd_bwd(self.h, _p(al), _p(be), _p(tot)))
        return al, be, tot

    # -- python views used by the parity tests ---------------------------------
    def segment(self, **o):
        self.run(SEGMENT, **o)
        off, w, t0, t1, lp = self.fetch_segment()
        return [list(zip(w[a:b].tolist(), t0[a:b].tolist(), t1[a:b].tolist(), lp[a:b].tolist()))
                for a, b in zip(off[:-1], off[1:])]

    def position(self, **o):
        self.run(POSITION, **o)
        off, w, p, t0, t1, lp = self.fetch_position()
        return [list(zip(w[a:b].tolist(), p[a:b].tolist(), t0[a:b].tolist(), t1[a:b].tolist(), lp[a:b].tolist()))
                for a, b in zip(off[:-1], off[1:])]

    def utterance(self, **o):
        self.run(UTTERANCE, **o)
        off, w, lp = self.fetch_utterance()
        return [list(zip(w[a:b].tolist(), lp[a:b].tolist())) for a, b in zip(off[:-1], off[1:])]

    def frame_post(self, **o):
        self.run(FRAME_POST, **o)
        off, nf, fr, w, lp = self.fetch_frame_post()
        res = []
        for l, (a, b) in enumerate(zip(off[:-1], off[1:])):
            frames = [[] for _ in range(int(nf[l]))]
            for k, ww, p in zip(fr[a:b].tolist(), w[a:b].tolist(), lp[a:b].tolist()):
                frames[k].append((ww, p))
            res.append(frames)
        return res

    def frame_post_csr(self, **o):
        """frame_post() through klu_fetch_frame_post_csr (no per-row frame column)."""
        self.run(FRAME_POST, **o)
        off, nf, fo, w, lp = self.fetch_frame_post_csr()
        res, slot = [], 0
        for l, (a, b) in enumerate(zip(off[:-1], off[1:])):
            T = int(nf[l])
            fl = fo[slot:slot + T + 1]
            slot += T + 1
            assert int(fl[T]) == int(b - a)
            res.append([list(zip(w[a + int(fl[k]):a + int(fl[k + 1])].tolist(), lp[a + int(fl[k]):a + int(fl[k + 1])].tolist()))
                        for k in range(T)])
        return res

    def position_post(self, **o):
        """Per lattice: list (one per transcript position) of lists of (word, float32 logp)."""
        self.run(POSITION_POST, **o)
        off, npos, pos, w, lp = self.fetch_position_post()
        res = []
        for l, (a, b) in enumerate(zip(off[:-1], off[1:])):
            rows = [[] for _ in range(int(npos[l]))]
            for k, ww, p in zip(pos[a:b].tolist(), w[a:b].tolist(), lp[a:b].tolist()):
                rows[k].append((ww, p))
            res.append(rows)
        return res

    def length_dist(self, **o):
        """Per lattice: [(length, float32 logp)] in the reference's output order."""
        self.run(LENGTH_DIST, **o)
        off = self.offsets()
        n = int(off[-1])
        ln, lp = np.zeros(n, np.int32), np.zeros(n, np.float32)
        _chk(self.L.klu_fetch_length_dist(self.h, _p(ln), _p(lp)))
        return [list(zip(ln[a:b].tolist(), lp[a:b].tolist())) for a, b in zip(off[:-1], off[1:])]

    def best_path2(self, **o):
        self.run(BEST_PATH2, **o)
        off, lab, cost, nf = self.fetch_best_path2()
        return [(lab[a:b].tolist(), float(cost[l])) for l, (a, b) in enumerate(zip(off[:-1], off[1:]))]

    def prune_arcs(self, **o):
        """lattice-prune-arcs: like prune_dyn_beam(); `first_kept` / `cutoff` instead of the beams."""
        self.run(PRUNE_ARCS, **o)
        res = self._pruned_lattices()
        for r in res:
            r["cutoff"], r["first_kept"] = r.pop("beam0"), int(r.pop("beam"))
        return res

    def prune_dyn_beam(self, **o):
        self.run(PRUNE_DYN_BEAM, **o)
        return self._pruned_lattices()

    def _pruned_lattices(self):
        off, ai, ns, nd, g, a, smap, fg, fa, beams = self.fetch_prune()
        b = self.batch
        res = []
        for l, (x, y) in enumerate(zip(off[:-1], off[1:])):
            s0, s1 = int(b.state_off[l]), int(b.state_off[l + 1])
            e0 = int(b.arc_off[l])
            arcs = [(int(ai[k]), int(ns[k]), int(nd[k]), int(b.label[e0 + ai[k]]), float(g[k]), float(a[k]))
                    for k in range(x, y)]
            m = smap[s0:s1]
            finals = [(int(m[s]), float(fg[s0 + s]), float(fa[s0 + s])) for s in range(s1 - s0)
                      if m[s] >= 0 and not (np.isinf(fg[s0 + s]) and np.isinf(fa[s0 + s]))]
            res.append(dict(arcs=arcs, finals=finals, nstates=int((m >= 0).sum()), beam0=float(beams[2 * l]),
                            beam=float(beams[2 * l + 1])))
        return res

    def pruned_batch(self):
        """The lattices lattice-prune-dyn-beam would write, as a LatticeBatch (numpy only): the
        input of the second stage of BASELINE.json configs[2] (prune piped into best-path2)."""
        from .lattice import LatticeBatch
        off, ai, ns, nd, g, a, smap, fg, fa, beams = self.fetch_prune()
        b = self.batch
        L = len(b)
        keep = smap >= 0
        lat_of_state = np.repeat(np.arange(L), np.diff(b.state_off))
        so = np.zeros(L + 1, np.int64)
        np.cumsum(np.bincount(lat_of_state[keep], minlength=L), out=so[1:])
        lat_of_arc = np.repeat(np.arange(L), np.diff(off))
        orig = b.arc_off[lat_of_arc] + ai
        return LatticeBatch(list(b.keys), so, off.astype(np.int64), np.ascontiguousarray(ns), np.ascontiguousarray(nd),
                            np.ascontiguousarray(b.label[orig]), np.ascontiguousarray(b.dur[orig]),
                            np.ascontiguousarray(g), np.ascontiguousarray(a), np.ascontiguousarray(fg[keep]),
                            np.ascontiguousarray(fa[keep]), np.ascontiguousarray(b.fin_dur[keep]))

    def char_position(self, wspace, other_groups=(), **o):
        lg, inc, dele = char_groups(wspace, other_groups)
        self.run(CHAR_POSITION, label_group=lg, inc_groups=inc, del_groups=dele, **o)
        off, coff, chars, pos, t0, t1, lp = self.fetch_char_position()
        res = []
        for a, b in zip(off[:-1], off[1:]):
            rows = []
            for i in range(a, b):
                s = "_".join(str(c) for c in chars[coff[i]:coff[i + 1]].tolist())
                rows.append((s, int(pos[i]), int(t0[i]), int(t1[i]), float(lp[i])))
            res.append(rows)
        return res

    def char_segment(self, wspace, other_groups=(), **o):
        """lattice-char-index-segment rows per lattice: (string, t0, t1, logp)."""
        lg, inc, dele = char_groups(wspace, other_groups)
        self.run(CHAR_SEGMENT, label_group=lg, inc_groups=inc, del_groups=dele, **o)
        off = self.offsets()
        n = int(off[-1])
        tot = C.c_int64()
        _chk(self.L.klu_result_char_sizes(self.h, C.byref(tot)))
        coff = np.zeros(n + 1, np.int64)
        chars = np.zeros(tot.value, np.int32)
        t0, t1 = np.zeros(n, np.int32), np.zeros(n, np.int32)
        lp = np.zeros(n, np.float64)
        _chk(self.L.klu_fetch_char_segment(self.h, _p(coff), _p(chars), _p(t0), _p(t1), _p(lp)))
        res = []
        for a, b in zip(off[:-1], off[1:]):
            res.append([("_".join(str(c) for c in chars[coff[i]:coff[i + 1]].tolist()), int(t0[i]), int(t1[i]),
                         float(lp[i])) for i in range(a, b)])
        return res

    def char_utterance(self, wspace, other_groups=(), **o):
        """lattice-char-index-utterance rows per lattice: (string, logp), logp = log P(the pseudo-word
        occurs at least once in the line), ordered by (logp desc, string asc)."""
        lg, inc, dele = char_groups(wspace, other_groups)
        self.run(CHAR_UTTERANCE, label_group=lg, inc_groups=inc, del_groups=dele, **o)
        off = self.offsets()
        n = int(off[-1])
        tot = C.c_int64()
        _chk(self.L.klu_result_char_sizes(self.h, C.byref(tot)))
        coff = np.zeros(n + 1, np.int64)
        chars = np.zeros(tot.value, np.int32)
        lp = np.zeros(n, np.float64)
        _chk(self.L.klu_fetch_char_utterance(self.h, _p(coff), _p(chars), _p(lp)))
        return [[("_".join(str(c) for c in chars[coff[i]:coff[i + 1]].tolist()), float(lp[i])) for i in range(a, b)]
                for a, b in zip(off[:-1], off[1:])]

    # -- measurement ------------------------------------------------------------
    def timer_start(self):
        _chk(self.L.klu_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        _chk(self.L.klu_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def launch_count(self):
        n = C.c_int64()
        _chk(self.L.klu_launch_count(self.h, C.byref(n)))
        return n.value

    def profile(self, on):
        _chk(self.L.klu_profile_enable(self.h, 1 if on else 0))

    def profile_json(self):
        buf = C.create_string_buffer(1 << 16)
        _chk(self.L.klu_profile_json(self.h, buf, C.c_size_t(len(buf))))
        return json.loads(buf.value.decode())

    def stats(self):
        s = (C.c_int64 * 8)()
        _chk(self.L.klu_batch_stats(self.h, s))
        return dict(lattices=s[0], states=s[1], arcs=s[2], levels=s[3], entries=s[4], band=s[5], frame_instances=s[6],
                    max_time=s[7])

    def load_times(self):
        """(upload ms, device packer ms, frame index ms) of the last load (klu_load_times)."""
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        _chk(self.L.klu_load_times(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def flush_l2(self):
        _chk(self.L.klu_flush_l2(self.h))
