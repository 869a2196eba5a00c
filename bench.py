#!/usr/bin/env python
"""bench.py -- lattice arcs/sec through the forward-backward + posterior-index hot path on
B200 (metric of BASELINE.json), with roofline, pack time, per-tool numbers and CPU baselines.

  python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
  python bench.py --impl reference --gpus N --steps K ...  (reference arm: the CPU
      restatement of the reference's algorithm -- oracle/ -- on all host threads;
      the reference itself needs Kaldi+OpenFst and cannot be built in this image)

The headline line is BASELINE.json configs[1]: lattice-to-word-frame-post with
--acoustic-scale=0.1 on 10k synthetic lattices PER GPU (~2k states / ~50k arcs each, 50k
vocabulary; weak scaling: lattices are independent, every rank owns its own shard, no
collective on the data path).

  value            arcs/s of a "step" = {alpha sweep, beta sweep, per-frame group sums of the
                   arc posteriors, per-frame ordering} with the packed batch AND its frame
                   index resident in HBM.  The sort of the arc x frame instances by
                   (frame, word) is NOT in this step: it depends on the lattice structure
                   only and runs once per batch, in the device packer -- see pack_ms.
  pack_ms          CUDA-event time of what the device does once per batch before the first
                   step: the packer of klu_load (levels, CSR, bands) + the frame index.
  value_incl_pack  arcs/s with pack_ms added to every step: the figure for a tool that
                   loads a batch and runs it once (what the drop-in binaries do).
  e2e              klu_load (H2D of the caller's pinned SoA arrays + packer) + klu_run +
                   klu_fetch_* (D2H of the whole index) through the C ABI, wall clock.
  tools            the other tools of BASELINE.json's configs, one entry each (N = 1 only):
                   ms per step, arcs/s, pack_ms, their own byte model, a bounded CPU baseline.
  --scaling strong one fixed batch partitioned by arc count over the ranks (shard.py).
  --dump-outputs   what the last timed step computed, as .npy files (dump_outputs()): the inputs
                   are seeded, so two builds run with the same arguments compare output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402

TOOLS = {"frame_post": 3, "segment": 0, "position": 1, "utterance": 2, "fwd_bwd": 7, "prune_dyn_beam": 4,
         "best_path2": 5, "position_post": 8, "char_position": 6, "prune_arcs": 11}
METRIC = "lattice arcs/sec (fwd-bwd + word-position index)"  # BASELINE.json's metric name, kept verbatim
METRIC_NOTE = ("`value` is measured on BASELINE.json configs[1] (lattice-to-word-frame-post, the configuration the "
               "metric is quoted on); the word-position index tool itself (lattice-word-index-position) is "
               "tools['position@c2']")
# algorithmic HBM bytes (SURVEY.md 8d): per arc / per state / per emitted entry
ALGO = {
    # alpha sweep src+g+a (12) + beta sweep dst+g+a (12); alpha+beta written once (16/state)
    "k_log_sweeps": dict(arc=24.0, state=16.0, entry=0.0),
    "k_banded_alpha": dict(arc=0.0, state=0.0, entry=0.0, band=8.0, unfolded=12.0),
    "k_pos_cells": dict(arc=0.0, state=0.0, entry=16.0, unfolded=20.0),
    "k_emit": dict(arc=20.0, state=0.0, entry=16.0),
    "k_seg_radix_sort": dict(arc=0.0, state=0.0, entry=16.0),
    "k_reduce": dict(arc=0.0, state=0.0, entry=16.0),
    "k_count_scan": dict(arc=8.0, state=0.0, entry=0.0),
    "k_gather": dict(arc=0.0, state=0.0, entry=16.0),
    # per-frame ordering: 4 B logp + 4 B word read, (word, logp) written in order (the frame column is static)
    "k_frame_order": dict(arc=0.0, state=0.0, entry=16.0),
    # fused window kernel: record + source id per arc (20 B), arc id per instance (4 B), offset read +
    # log-posterior written per group (8 B)
    "k_frame_groups": dict(arc=20.0, state=16.0, entry=8.0, inst=4.0),
    "k_trop_sweeps": dict(arc=24.0, state=16.0, entry=0.0),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons DURING the timed region: NVML in-process
    (a few ms per sample); nvidia-smi subprocesses only if NVML is unavailable."""

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.stop_flag, self.samples, self.reasons, self.max_mhz = gpu, False, [], set(), None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        n = self.nvml
        self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(
            n, "nvmlDeviceGetCurrentClocksEventReasons") else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                          ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5)
        f = [x.strip() for x in out.stdout.strip().split(",")]
        self.samples.append(float(f[0]))
        self.max_mhz = float(f[1])
        for n, v in zip(names, f[2:]):
            if v.lower().startswith("active"):
                self.reasons.add(n)

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.sample_nvml()
                else:
                    self.sample_smi()
            except Exception:
                pass
            time.sleep(0.005 if self.nvml is not None else 0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def numa_bind(local):
    """Pins this rank (and the pinned buffers it is about to allocate: first touch) to the CPUs of the
    NUMA node its GPU hangs off, so 8 ranks' uploads do not all cross one socket's memory controller.
    Best effort (sysfs only); returns what it did for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return {"node": None, "note": "no NUMA affinity reported for %s" % bdf}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"node": node, "note": "node has no CPU this process may use"}
        os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus), "pci": bdf}
    except Exception as ex:  # no sysfs / no torch attribute: leave the affinity alone
        return {"node": None, "note": "%s: %s" % (type(ex).__name__, ex)}


def dist_setup(n):
    """Returns (rank, world, reduce_max, barrier, gather_obj)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world == 1:
        return 0, 1, (lambda x: x), (lambda: None), (lambda x: [x])
    import torch
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    def gather_obj(x):
        out = [None] * world
        dist.all_gather_object(out, x)
        return out

    return rank, world, reduce_max, barrier, gather_obj


def flags_for(tool):
    if tool == "prune_dyn_beam":  # BASELINE.json configs[2]
        return dict(max_arcs=20000, max_states=1500, beam_ratio=0.9)
    if tool == "char_position":
        return dict(nbest=100)
    if tool == "prune_arcs":
        return dict(acoustic_scale=0.1, beam=0.5)
    return dict(acoustic_scale=0.1)


def run_tool(eng, klu, tool, flags):
    if tool == "char_position":
        lg, inc, dele = klu.binding.char_groups([1], ())
        o, keep = klu.binding.make_opts(label_group=lg, inc_groups=inc, del_groups=dele, **flags)
        eng.run_opts(klu.CHAR_POSITION, o)
    else:
        eng.run(TOOLS[tool], **flags)


def fetch_arrays(eng, klu, tool, out=None):
    """The arrays the last run of `tool` hands to a caller (klu_fetch_*)."""
    t = TOOLS[tool]
    if t == klu.FRAME_POST:
        # the rows as the reference's Posterior holds them: per-frame row offsets instead of a frame column
        return eng.fetch_frame_post_csr(out=out)
    if t == klu.SEGMENT:
        return eng.fetch_segment()
    if t == klu.POSITION:
        return eng.fetch_position()
    if t == klu.POSITION_POST:
        return eng.fetch_position_post()
    if t == klu.UTTERANCE:
        return eng.fetch_utterance()
    if t == klu.FWD_BWD:
        return eng.fetch_fwd_bwd()
    if t in (klu.PRUNE_DYN_BEAM, klu.PRUNE_ARCS):
        return eng.fetch_prune()
    if t == klu.BEST_PATH2:
        return eng.fetch_best_path2()
    if t == klu.CHAR_POSITION:
        return eng.fetch_char_position()
    raise ValueError(tool)


def fetch_for(eng, klu, tool, out=None):
    """(rows, bytes brought to the host) of the last run."""
    r = fetch_arrays(eng, klu, tool, out)
    rows = 0 if TOOLS[tool] == klu.FWD_BWD else int(r[0][-1])
    return rows, sum(int(x.nbytes) for x in r)


def time_steps(eng, klu, tool, flags, steps, warmup):
    for _ in range(warmup):
        run_tool(eng, klu, tool, flags)
    eng.sync()
    eng.timer_start()
    for _ in range(steps):
        run_tool(eng, klu, tool, flags)
    return eng.timer_stop() / steps


DUMP_BYTES = 63 * 10**6  # under 64 MB with the .npy headers
DUMP_LATTICES = 64


def dump_outputs(eng, klu, tool, batch, d):
    """Writes what the last run of `tool` hands to a caller as DIR/<name>.npy: the per-lattice arrays of
    the whole batch, and the per-row / per-state arrays of a fixed, seeded sample of lattices (at most 64,
    fewer where their rows would take the files past 64 MB; `sample.npy` lists them).  Floats keep their
    dtype, integers are stored as float64 (exact).  Returns (sampled lattices, bytes written)."""
    nlat = len(batch)
    t = TOOLS[tool]
    r = fetch_arrays(eng, klu, tool)
    if t == klu.FWD_BWD:
        al, be, tot = r
        whole = {"total": tot}
        parts = {"alpha": (al, batch.state_off), "beta": (be, batch.state_off)}
    else:
        off = r[0]
        whole = {"rows": np.diff(off)}

        def by_row(names, xs):
            return {k: (x, off) for k, x in zip(names, xs)}

        if t == klu.FRAME_POST:
            _, nf, fo, w, lp = r
            whole["num_frames"] = nf
            slots = np.concatenate([[0], np.cumsum(nf.astype(np.int64) + 1)])
            parts = {"frame_row_off": (fo, slots), "word": (w, off), "logp": (lp, off)}
        elif t == klu.SEGMENT:
            parts = by_row(("word", "t0", "t1", "logp"), r[1:])
        elif t == klu.POSITION:
            parts = by_row(("word", "pos", "t0", "t1", "logp"), r[1:])
        elif t == klu.POSITION_POST:
            whole["num_pos"] = r[1]
            parts = by_row(("pos", "word", "logp"), r[2:])
        elif t == klu.UTTERANCE:
            parts = by_row(("word", "logp"), r[1:])
        elif t == klu.BEST_PATH2:
            whole["cost"], whole["num_frames"] = r[2], r[3]
            parts = by_row(("label",), r[1:2])
        elif t in (klu.PRUNE_DYN_BEAM, klu.PRUNE_ARCS):
            _, ai, ns, nd, g, a, smap, fg, fa, beams = r
            whole["beams"] = beams.reshape(nlat, 2)
            parts = by_row(("arc", "src", "dst", "graph", "acoustic"), (ai, ns, nd, g, a))
            per_state = zip(("state_map", "fin_graph", "fin_acoustic"), (smap, fg, fa))
            parts.update({k: (x, batch.state_off) for k, x in per_state})
        elif t == klu.CHAR_POSITION:
            _, coff, chars, pos, t0, t1, lp = r
            parts = by_row(("num_chars", "pos", "t0", "t1", "logp"), (np.diff(coff), pos, t0, t1, lp))
            parts["chars"] = (chars, coff[off])
        else:
            raise ValueError(tool)

    def out(x):
        return x if x.dtype in (np.float32, np.float64) else x.astype(np.float64)

    budget = DUMP_BYTES - sum(out(x).nbytes for x in whole.values()) - 8 * min(nlat, DUMP_LATTICES)
    cost = np.zeros(nlat, np.int64)
    for x, o in parts.values():
        cost += np.diff(np.asarray(o, np.int64)) * out(x[:0]).itemsize
    order = np.random.RandomState(0x5EED).permutation(nlat)[:DUMP_LATTICES]
    sample = np.sort(order[:int(np.searchsorted(np.cumsum(cost[order]), budget, side="right"))])
    files = {k: out(np.asarray(x)) for k, x in whole.items()}
    files["sample"] = sample.astype(np.float64)
    for k, (x, o) in parts.items():
        files[k] = out(np.concatenate([x[:0]] + [x[int(o[l]):int(o[l + 1])] for l in sample]))
    os.makedirs(d, exist_ok=True)
    for k, x in files.items():
        np.save(os.path.join(d, k + ".npy"), x)
    return len(sample), sum(x.nbytes for x in files.values())


def kernel_profile(eng, klu, tool, flags, runs=2):
    eng.profile(True)
    for _ in range(runs):
        run_tool(eng, klu, tool, flags)
    prof = eng.profile_json()
    eng.profile(False)
    return {k: {"launches_per_step": v["launches"] / runs, "ms_per_step": v["ms"] / runs} for k, v in prof.items()}


def oracle_tool(ora, tool):
    return {"frame_post": ora.FRAME_POST, "segment": ora.SEGMENT, "position": ora.POSITION,
            "utterance": ora.UTTERANCE, "best_path2": ora.BEST_PATH2, "prune_dyn_beam": ora.PRUNE_DYN_BEAM,
            "position_post": ora.POSITION_POST}[tool]


def run_reference(args, rank, world):
    """Reference arm: CPU restatement on all host threads, bounded sample."""
    if rank != 0:
        return
    klu = load_package()
    from oracle import ora
    ora.build()
    cores = os.cpu_count() or 1
    n = args.ref_lattices
    batch = klu.synth_batch(args.shape, n, seed=args.seed)
    lats = batch.lattices()
    tool = oracle_tool(ora, args.tool)
    for _ in range(min(args.warmup, 1)):
        ora.run_batch(tool, lats[:cores], cores, **flags_for(args.tool))
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        ora.run_batch(tool, lats, cores, **flags_for(args.tool))
        times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    v = batch.num_arcs / sec
    sample = "%d lattices of the workload (%d arcs) per step, %d host threads" % (n, batch.num_arcs, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v,
        "unit": "arcs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(args, args.lattices),
        "cpu_baseline": {"value": v, "unit": "arcs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "arcs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def workload_config(args, nlat):
    return {"workload": "BASELINE.json configs[1]: lattice-to-word-frame-post forward-backward on %d synthetic "
                        "lattices per GPU (~2k states, ~50k arcs, 50k vocab), --acoustic-scale=0.1" % nlat
            if args.tool == "frame_post" and args.shape == "c2" else
            "%s on %d synthetic '%s' lattices per GPU" % (args.tool, nlat, args.shape),
            "tool": args.tool, "shape": args.shape, "lattices_per_gpu": nlat, "seed": args.seed,
            "l2_policy": "inputs (packed arcs, >10 GB) far larger than the 126 MB L2; no explicit flush",
            "parallelism": "independent lattice shards per GPU, no collective"}


# ------------------------------------------------------------------ per-tool section ---
def model_bytes(tool, st, entries, unfolded):
    """Algorithmic HBM bytes of one step (SURVEY.md 8d)."""
    arcs, states = st["arcs"], st["states"]
    if tool in ("segment", "utterance"):
        # alpha 12 + beta 12 + emit read 20 + emit write 16 + reduce read 16 per arc; 28 per state
        return 76.0 * arcs + 28.0 * states, "76 B/arc + 28 B/state"
    if tool in ("position", "best_path2", "position_post"):
        # fwd-bwd (24 B/arc + 16 B/state) + per arc of the length-unfolded lattice (E x I_L): banded
        # sweep 12, emit read 20 + write 16, reduce read 16; 8 B per (state, length) cell written
        return (24.0 * arcs + 16.0 * states + 64.0 * unfolded + 8.0 * st["band"],
                "24 B/arc + 16 B/state + 64 B/unfolded arc + 8 B/(state,len) cell")
    if tool == "prune_dyn_beam":
        return 37.0 * arcs + 16.0 * states, "37 B/arc + 16 B/state"
    if tool == "fwd_bwd":
        return 24.0 * arcs + 16.0 * states, "24 B/arc + 16 B/state"
    return None, None


def unfolded_arcs(batch):
    """Arcs of the length-unfolded lattice, sum over arcs of the source state's number of
    distinct label counts (E x I_L of SURVEY.md 8d): a forward DP over (min, max) label
    counts per state, exact when every count in between is reachable (true of the shapes here)."""
    total = 0
    for l in range(len(batch)):
        s0, s1 = int(batch.state_off[l]), int(batch.state_off[l + 1])
        e0, e1 = int(batch.arc_off[l]), int(batch.arc_off[l + 1])
        n = s1 - s0
        src, dst, nz = batch.src[e0:e1], batch.dst[e0:e1], (batch.label[e0:e1] != 0).astype(np.int64)
        lo = np.full(n, 1 << 40, np.int64)
        hi = np.full(n, -1, np.int64)
        if n:
            lo[0] = hi[0] = 0
        first = np.searchsorted(src, np.arange(n + 1))
        for s in range(n):
            a, b = first[s], first[s + 1]
            if b > a and hi[s] >= 0:
                np.minimum.at(lo, dst[a:b], lo[s] + nz[a:b])
                np.maximum.at(hi, dst[a:b], hi[s] + nz[a:b])
        w = np.where(hi >= 0, hi - lo + 1, 0)
        total += int(w[src][batch.label[e0:e1] != 0].sum())
    return total


def cpu_sample(klu, ora, tool, batch, n, flags, cores, **extra):
    sub = batch.slice(0, min(n, len(batch)))
    t0 = time.perf_counter()
    ora.run_batch(oracle_tool(ora, tool), sub.lattices(), cores, **flags, **extra)
    dt = time.perf_counter() - t0
    return sub, dt


def char_tool_entry(args, shape, nlat, ncpu, cores, local):
    last = None
    for attempt in range(3):
        cmd = [sys.executable, os.path.abspath(__file__), "--tool", "char_position", "--shape", shape, "--lattices",
               str(nlat), "--steps", str(args.tools_steps), "--warmup", "3", "--e2e-steps", "0", "--no-tools",
               "--ref-lattices", str(ncpu), "--seed", str(args.seed)] + (["--no-cpu-baseline"] if args.no_cpu_baseline else [])
        env = dict(os.environ, LOCAL_RANK=str(local))
        for k in ("RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
            line = [x for x in r.stdout.splitlines() if x.startswith("{")]
            if r.returncode == 0 and line:
                d = json.loads(line[-1])
                return {"tool": "char_position", "shape": shape, "lattices": nlat, "arcs": d["batch"]["arcs"],
                        "states": d["batch"]["states"], "flags": flags_for("char_position"), "ms_per_step": d["ms_per_step"],
                        "arcs_per_s": d["value"], "pack_ms": d["pack_ms"], "arcs_per_s_incl_pack": d["value_incl_pack"],
                        "index_entries": d["batch"]["index_entries"],
                        "kernels_ms": {k: round(v["ms_per_launch"] * v["launches_per_step"], 3)
                                       for k, v in d["roofline"]["kernels"].items()},
                        "cpu_baseline": d["cpu_baseline"], "attempts": attempt + 1, "own_process": True}
            last = (r.stderr or r.stdout).strip().splitlines()[-1:] or ["rc=%d" % r.returncode]
        except Exception as ex:
            last = ["%s: %s" % (type(ex).__name__, ex)]
    return {"error": last[0] if last else "failed", "attempts": 3}


def bench_tools(klu, local, args, peak):
    """Device-resident numbers of the other tools named by BASELINE.json's configs, each with
    its pack time, byte model and a bounded CPU baseline (oracle port on all host threads)."""
    from oracle import ora
    ora.build()
    cores = os.cpu_count() or 1
    out = {}
    specs = [("segment@c2", "segment", "c2", args.tools_scale * 3000, 256),
             ("position@c2", "position", "c2", args.tools_scale * 256, cores),
             ("utterance@c4", "utterance", "c4", args.tools_scale * 32, cores),
             ("prune_dyn_beam->best_path2@c2", "prune_dyn_beam", "c2", args.tools_scale * 1024, 2 * cores),
             ("char_position@c5", "char_position", "c5", args.tools_scale * 256, 2 * cores)]
    for name, tool, shape, nlat, ncpu in specs:
        nlat = int(max(1, nlat))
        if tool == "char_position":
            # The character tool runs in a process of its own, up to three times, at the batch size
            # the drop-in binaries use for it (256 lattices): before the merge kernel and the sorts
            # were rewritten, batches of 448+ c5 lattices (trie frontier past 3e8 candidates at one
            # depth) ended in an illegal memory access in 2 runs of 5 (DESIGN.md "known issues"; not
            # seen since in 14 runs), which would take this process's CUDA context with it.
            out[name] = char_tool_entry(args, shape, nlat, ncpu, cores, local)
            continue
        eng = klu.Engine(local)
        try:
            t0 = time.perf_counter()
            batch = klu.synth_batch(shape, nlat, seed=args.seed)
            flags = flags_for(tool)
            eng.load(batch)
            eng.load(batch)  # the second load's times: no first-use cudaMalloc inside the events
            up_ms, pack_ms, _ = eng.load_times()
            st = eng.stats()
            ms = time_steps(eng, klu, tool, flags, args.tools_steps, 2)
            entries, _ = fetch_for(eng, klu, tool)
            kern = kernel_profile(eng, klu, tool, flags, 1)
            entry = {"tool": tool, "shape": shape, "lattices": nlat, "arcs": st["arcs"], "states": st["states"],
                     "flags": flags, "ms_per_step": ms, "arcs_per_s": st["arcs"] / (ms * 1e-3), "pack_ms": pack_ms,
                     "arcs_per_s_incl_pack": st["arcs"] / ((ms + pack_ms) * 1e-3), "index_entries": entries,
                     "kernels_ms": {k: round(v["ms_per_step"], 3) for k, v in kern.items()}}
            unf = unfolded_arcs(batch.slice(0, min(8, nlat))) * (st["arcs"] / max(1, batch.slice(0, min(8, nlat)).num_arcs)) \
                if tool == "position" else 0
            if tool == "position":
                entry["unfolded_arcs"] = unf
            mb, mdesc = model_bytes(tool, st, entries, unf)
            if mb:
                entry["model"] = mdesc
                entry["model_bytes_per_step"] = mb
                entry["hbm_frac"] = mb / (ms * 1e-3) / 1e9 / peak
            # ---- second stage of configs[2]: lattice-best-path2 on the pruned lattices
            if tool == "prune_dyn_beam":
                pruned = eng.pruned_batch()
                eng.load(pruned)
                eng.load(pruned)
                _, pack2, _ = eng.load_times()
                f2 = dict()
                ms2 = time_steps(eng, klu, "best_path2", f2, args.tools_steps, 2)
                st2 = eng.stats()
                entry.update({"ms_prune": ms, "ms_best_path2": ms2, "pruned_arcs": st2["arcs"], "ms_per_step": ms + ms2,
                              "pack_ms": pack_ms + pack2, "arcs_per_s": st["arcs"] / ((ms + ms2) * 1e-3),
                              "arcs_per_s_incl_pack": st["arcs"] / ((ms + ms2 + pack_ms + pack2) * 1e-3)})
                entry.pop("hbm_frac", None)
            # ---- CPU baseline: bounded sample on all host threads
            if not args.no_cpu_baseline:
                if tool == "utterance":
                    # the reference composes the lattice with a query automaton per word (~40k words x
                    # 500k arcs per c4 lattice: tens of minutes per lattice): a sample of words through
                    # --include-words, scaled to all words
                    lat0 = batch[0]
                    words = np.unique(lat0.label[lat0.label != 0])
                    pick = np.random.RandomState(1).choice(words, min(48, len(words)), replace=False).tolist()
                    sub, dt = cpu_sample(klu, ora, tool, batch, ncpu, flags, cores, include_words=pick)
                    done = sum(int(np.isin(np.unique(l.label), pick).sum()) for l in sub.lattices())
                    allw = sum(int(np.unique(l.label[l.label != 0]).size) for l in sub.lattices())
                    dt_full = dt * allw / max(1, done)
                    entry["cpu_baseline"] = {"value": sub.num_arcs / dt_full, "unit": "arcs/s", "cores": cores, "kind": "port",
                                             "sample": "first %d lattices, %d of their %d (lattice, word) queries run "
                                                       "(--include-words) in %.1f s on %d threads, scaled to all words"
                                                       % (len(sub), done, allw, dt, cores), "extrapolated": True}
                elif tool == "prune_dyn_beam":
                    sub, dt = cpu_sample(klu, ora, tool, batch, ncpu, flags, cores)
                    sub2 = pruned.slice(0, len(sub))
                    t0b = time.perf_counter()
                    ora.run_batch(ora.BEST_PATH2, sub2.lattices(), cores)
                    dt2 = time.perf_counter() - t0b
                    entry["cpu_baseline"] = {"value": sub.num_arcs / (dt + dt2), "unit": "arcs/s", "cores": cores,
                                             "kind": "port", "sample": "first %d lattices: prune %.1f s + best-path2 on "
                                             "the pruned lattices %.1f s, %d threads" % (len(sub), dt, dt2, cores)}
                else:
                    sub, dt = cpu_sample(klu, ora, tool, batch, ncpu, flags, cores)
                    entry["cpu_baseline"] = {"value": sub.num_arcs / dt, "unit": "arcs/s", "cores": cores, "kind": "port",
                                             "sample": "first %d lattices, %.1f s on %d threads" % (len(sub), dt, cores)}
            entry["wall_s"] = round(time.perf_counter() - t0, 1)
            out[name] = entry
        except Exception as ex:  # one tool failing must not lose the headline line
            out[name] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        finally:
            eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tool", default="frame_post", choices=sorted(TOOLS))
    ap.add_argument("--shape", default="c2")
    ap.add_argument("--lattices", type=int, default=10000, help="lattices per GPU (weak) / in total (strong)")
    ap.add_argument("--ref-lattices", type=int, default=2500, help="bounded CPU sample (lattices) per step")
    ap.add_argument("--seed", type=int, default=0x5EED)
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-slices", type=int, default=16, help="slices of the pipelined end-to-end run (1 = off)")
    ap.add_argument("--e2e-contexts", type=int, default=8, help="contexts (host threads) of the pipelined run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-tools", action="store_true", help="skip the per-tool section")
    ap.add_argument("--tools-steps", type=int, default=3)
    ap.add_argument("--tools-scale", type=float, default=1.0, help="scales the per-tool lattice counts")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's shard) as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm counts rows and returns no arrays")

    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        run_reference(args, rank, int(os.environ.get("WORLD_SIZE", "1")))
        return

    rank, world, reduce_max, barrier, gather_obj = dist_setup(args.gpus)
    klu = load_package()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    all_cpus = os.sched_getaffinity(0)
    numa = numa_bind(local) if not os.environ.get("KLU_BENCH_NO_NUMA") else {"node": None, "note": "disabled"}
    eng = klu.Engine(local)
    tool = TOOLS[args.tool]
    flags = flags_for(args.tool)

    # ---- this rank's lattices, generated straight into pinned host memory
    keep = []

    def alloc(nbytes):
        buf = eng.pinned(nbytes)
        keep.append(buf)
        return buf

    t0 = time.perf_counter()
    strong = None
    if args.scaling == "strong" and world > 1:
        # ONE batch of --lattices lattices for the whole job, cut by total arc count with the
        # product's partitioner (shard.partition_by_arcs: greedy longest-first); every rank
        # generates only its own lattices (the generator is deterministic in (seed, id))
        so = np.zeros(args.lattices + 1, np.int64)
        ao = np.zeros(args.lattices + 1, np.int64)
        cfg = klu.lattice.SynthCfg(**klu.lattice.SHAPES[args.shape])
        import ctypes as C
        klu.lattice.hostlib().klu_synth_sizes(C.byref(cfg), args.seed, 0, args.lattices, so.ctypes.data,
                                              ao.ctypes.data, min(os.cpu_count() or 1, 64))
        counts = np.diff(ao)
        shards = klu.partition_by_arcs(counts, world)
        mine = shards[rank]
        parts = [klu.synth_batch(args.shape, 1, seed=args.seed, first_id=i, nthreads=1) for i in mine]
        per = [int(counts[s].sum()) for s in shards]
        strong = {"total_lattices": args.lattices, "total_arcs": int(counts.sum()), "arcs_per_shard": per,
                  "imbalance_max_over_mean": max(per) / (sum(per) / len(per)), "partitioner": "shard.partition_by_arcs"}
        cat = klu.LatticeBatch.from_lattices([p[0] for p in parts])

        def pin(x):  # the shard's arrays in pinned host memory, like the generated ones
            buf = np.frombuffer(alloc(max(x.nbytes, 1)), dtype=x.dtype, count=x.size)
            buf[:] = x
            return buf

        batch = klu.LatticeBatch(cat.keys, cat.state_off, cat.arc_off, *[pin(getattr(cat, f)) for f in (
            "src", "dst", "label", "dur", "graph", "acoustic", "fin_graph", "fin_acoustic", "fin_dur")])
        nlat = len(batch)
    else:
        nlat = args.lattices
        batch = klu.synth_batch(args.shape, nlat, seed=args.seed, first_id=rank * nlat, alloc=alloc)
    t_gen = time.perf_counter() - t0
    t0 = time.perf_counter()
    eng.load(batch)
    t_load = time.perf_counter() - t0
    st = eng.stats()
    arcs, states = st["arcs"], st["states"]
    total_arcs = sum(gather_obj(arcs))

    # ---- device-resident timing (value) ----
    for _ in range(max(args.warmup, 3)):
        run_tool(eng, klu, args.tool, flags)
    eng.sync()
    up_ms, pack_ms, frame_ms = eng.load_times()  # the frame index is built by the first frame-post run
    pack_total = pack_ms + frame_ms
    launches0 = eng.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    eng.sync()
    eng.timer_start()
    for _ in range(args.steps):
        run_tool(eng, klu, args.tool, flags)
    ms = eng.timer_stop()
    barrier()
    sampler.stop_flag = True
    launches = eng.launch_count() - launches0
    ms = reduce_max(ms)
    ms_per_step = ms / args.steps
    pack_total = reduce_max(pack_total)
    entries, _ = fetch_for(eng, klu, args.tool)
    value = total_arcs / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        nsample, nbytes = dump_outputs(eng, klu, args.tool, batch, args.dump_outputs)
        sys.stderr.write("bench: outputs of the last timed step (%d sampled lattices, %d bytes) in %s\n"
                         % (nsample, nbytes, args.dump_outputs))

    # ---- per-kernel profile (CUDA events on the launching stream) ----
    prof = kernel_profile(eng, klu, args.tool, flags, 2)
    tot_ms = sum(v["ms_per_step"] for v in prof.values()) or 1.0
    dom = max(prof, key=lambda k: prof[k]["ms_per_step"])
    peak, peak_src = peaks()
    band = st["band"]
    unf = unfolded_arcs(batch.slice(0, min(8, nlat))) * (arcs / max(1, batch.slice(0, min(8, nlat)).num_arcs)) \
        if args.tool in ("position", "best_path2", "position_post") else 0

    def algo_bytes(name):
        a = ALGO.get(name, dict(arc=0, state=0, entry=0))
        return (a["arc"] * arcs + a["state"] * states + a["entry"] * entries + a.get("band", 0) * band +
                a.get("inst", 0) * st.get("frame_instances", 0) + a.get("unfolded", 0) * unf)

    kern = {}
    for k, v in prof.items():
        per_launch_ms = v["ms_per_step"] / max(v["launches_per_step"], 1e-9)
        ab = algo_bytes(k)
        kern[k] = {"launches_per_step": v["launches_per_step"], "ms_per_launch": per_launch_ms,
                   "share": v["ms_per_step"] / tot_ms,
                   "algo_GBps": ab / (v["ms_per_step"] * 1e-3) / 1e9 if v["ms_per_step"] > 0 else None}
    dom_ms = prof[dom]["ms_per_step"] / max(prof[dom]["launches_per_step"], 1e-9)
    achieved = algo_bytes(dom) / max(prof[dom]["launches_per_step"], 1e-9) / (dom_ms * 1e-3) / 1e9
    # whole-pipeline algorithmic model of SURVEY.md 8d: 76 B/arc + 28 B/state (the segment / position tools'
    # emit + reduce-by-key pipeline; quoted for the frame-post step only as a common yardstick)
    pipe_bytes = 76.0 * arcs + 28.0 * states
    traffic, traffic_note = None, None  # DRAM bytes per launch of the dominant kernel (ncu --set full)
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if dom in tj:
            traffic = tj[dom]["dram_bytes_per_arc"] * arcs
            traffic_note = tj[dom].get("note")
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes(dom) / max(prof[dom]["launches_per_step"], 1e-9),
                "pipeline_frac_76B_per_arc": pipe_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                "pipeline_frac_76B_per_arc_incl_pack": pipe_bytes / ((ms_per_step + pack_total) * 1e-3) / 1e9 / peak,
                "kernels": kern}

    # ---- end to end through the C ABI: host arrays -> index on the host ----
    # (a) one klu_load + klu_run + klu_fetch call sequence over the whole shard;
    # (b) the same calls pipelined the way the drop-in tools do it (KLU_DEVICES): the shard
    #     cut into slices by arc count, a few contexts on this GPU taking slices in turn, one
    #     host thread each, so that the upload of one slice overlaps packing, run and result
    #     download of the previous one.  `e2e.value` is (b); (a) is reported beside it.
    # the caller hands over per-state arc counts instead of a per-arc source array
    # (klu_lattices.state_num_arcs; OpenFst stores arcs grouped by state)
    narcs = batch.state_num_arcs()
    narcs_pinned = eng.pinned_array(np.int32, max(narcs.size, 1))
    narcs_pinned[:narcs.size] = narcs
    narcs = narcs_pinned[:narcs.size]
    # ... and durations as bytes / destinations as 16-bit distances from the source when they fit
    # (klu_lattices.arc_dur_u8 / arc_dst_delta_u16): 15 instead of 20 bytes per arc
    dur8, d16 = klu.binding.compact_arcs(batch)

    def pinned_copy(x):
        if x is None:
            return None
        buf = eng.pinned_array(x.dtype, max(x.size, 1))
        buf[:x.size] = x
        return buf[:x.size]

    # ... and labels as 16-bit words when the vocabulary allows (klu_lattices.arc_label_u16): 13 bytes per arc
    lab16 = klu.binding.compact_labels(batch)
    dur8, d16, lab16 = pinned_copy(dur8), pinned_copy(d16), pinned_copy(lab16)
    up = dict(state_num_arcs=narcs, dur_u8=dur8, dst_delta_u16=d16, label_u16=lab16)
    h2d = sum(int(x.nbytes) for x in (batch.state_off, batch.arc_off, narcs, d16 if d16 is not None else batch.dst,
                                      lab16 if lab16 is not None else batch.label, dur8 if dur8 is not None else batch.dur,
                                      batch.graph, batch.acoustic, batch.fin_graph, batch.fin_acoustic,
                                      batch.fin_dur))
    d2h = 0
    out = None
    if args.tool == "frame_post":  # results land in pinned host buffers
        nf_all = eng.fetch_frame_post_csr()[1].astype(np.int64)  # frames per lattice: sizes the row-offset array
        slot_off = np.concatenate([[0], np.cumsum(nf_all + 1)])
        out = (eng.pinned_array(np.int64, int(slot_off[-1])), eng.pinned_array(np.int32, entries),
               eng.pinned_array(np.float32, entries))
    e2e_ms, parts, packs = [], [], []
    for i in range(args.e2e_steps + 1 if args.e2e_steps > 0 else 0):
        barrier()
        t0 = time.perf_counter()
        eng.load(batch, **up)
        t1 = time.perf_counter()
        run_tool(eng, klu, args.tool, flags)
        eng.sync()
        t2 = time.perf_counter()
        _, d2h = fetch_for(eng, klu, args.tool, out)
        eng.sync()
        dt = time.perf_counter() - t0
        if i > 0:
            e2e_ms.append(1e3 * dt)
            parts.append((1e3 * (t1 - t0), 1e3 * (t2 - t1), 1e3 * (t0 + dt - t2)))
            packs.append(eng.load_times())
    single_step = reduce_max(sum(e2e_ms) / len(e2e_ms)) if e2e_ms else None
    if packs:  # pack time of a load with nothing else queued on the GPU (the e2e loads)
        pack_total = reduce_max(float(np.mean([p[1] + p[2] for p in packs])))
        roofline["pipeline_frac_76B_per_arc_incl_pack"] = pipe_bytes / ((ms_per_step + pack_total) * 1e-3) / 1e9 / peak
    pipe_step = None
    # contexts (host threads) per rank: no more than the host's cores divided among the ranks
    # (8 ranks x 8 spinning threads on a 32-core host get in each other's way); two slices per context
    n_ctx = args.e2e_contexts
    n_slices = args.e2e_slices
    if world > 1:
        n_ctx = max(3, min(n_ctx, len(all_cpus) // world))
        n_slices = min(n_slices, 2 * n_ctx) if n_ctx < args.e2e_contexts else n_slices
    if args.e2e_steps > 0 and n_slices > 1 and args.tool == "frame_post":
        eng.close()  # its device memory goes to the pipeline contexts
        nsl = min(n_slices, nlat)
        cuts = np.searchsorted(batch.arc_off, np.linspace(0, batch.arc_off[-1], nsl + 1)[1:-1]).tolist()
        cuts = [0] + [int(x) for x in cuts] + [nlat]
        subs = [batch.slice(a, b) for a, b in zip(cuts[:-1], cuts[1:])]
        sub_up = [dict(state_num_arcs=narcs[int(batch.state_off[a]):int(batch.state_off[b])],
                       dur_u8=None if dur8 is None else dur8[int(batch.arc_off[a]):int(batch.arc_off[b])],
                       dst_delta_u16=None if d16 is None else d16[int(batch.arc_off[a]):int(batch.arc_off[b])],
                       label_u16=None if lab16 is None else lab16[int(batch.arc_off[a]):int(batch.arc_off[b])])
                  for a, b in zip(cuts[:-1], cuts[1:])]
        engines = [klu.Engine(local) for _ in range(min(n_ctx, nsl))]
        row_off = np.concatenate([[0], np.cumsum([0] * nsl)])  # filled by the first pass
        sub_rows = [0] * nsl

        def work(k, record):
            e = engines[k]
            for j in range(k, nsl, len(engines)):
                e.load(subs[j], **sub_up[j])
                e.run(tool, **flags)
                if record:
                    sub_rows[j] = int(e.offsets()[-1])
                else:
                    a = int(row_off[j])
                    o = (out[0][int(slot_off[cuts[j]]):int(slot_off[cuts[j + 1]])], out[1][a:a + sub_rows[j]],
                         out[2][a:a + sub_rows[j]])
                    e.fetch_frame_post_csr(out=o)

        pipe_ms = []
        for i in range(args.e2e_steps + 2):
            barrier()
            t0 = time.perf_counter()
            th = [threading.Thread(target=work, args=(k, i == 0)) for k in range(len(engines))]
            for t in th:
                t.start()
            for t in th:
                t.join()
            dt = time.perf_counter() - t0
            if i == 0:
                row_off = np.concatenate([[0], np.cumsum(sub_rows)])
                assert int(row_off[-1]) == entries
            elif i > 1:
                pipe_ms.append(1e3 * dt)
        pipe_step = reduce_max(sum(pipe_ms) / len(pipe_ms))
        for e in engines:
            e.close()
    e2e_step = pipe_step if pipe_step else single_step
    e2e = {"value": total_arcs / (e2e_step * 1e-3) if e2e_step else None, "unit": "arcs/s",
           "ms_per_step": e2e_step, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "h2d_GBps_per_rank": h2d / (e2e_step * 1e-3) / 1e9 if e2e_step else None,
           "single_call_ms_per_step": single_step,
           "single_call_ms_load_run_fetch": [round(float(np.mean([p[k] for p in parts])), 2) for k in range(3)]
           if parts else None,
           "single_call_ms_upload_pack_frameindex": [round(float(np.mean([p[k] for p in packs])), 2) for k in range(3)]
           if packs else None,
           "pipeline": {"slices": n_slices, "contexts": n_ctx} if pipe_step else None,
           "note": "klu_load (H2D of the caller's pinned SoA arrays + device packer) + klu_run + klu_fetch "
                   "(D2H of the full index into pinned buffers), wall clock, max over ranks; value = the "
                   "pipelined call sequence when `pipeline` is set, else the single call sequence"}

    # ---- CPU baseline (rank 0, bounded sample of the same workload) ----
    os.sched_setaffinity(0, all_cpus)  # the CPU arms get every host thread again
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.tool == "char_position":
        from oracle import ora
        ora.build()
        cores = os.cpu_count() or 1
        sub = batch.slice(0, min(args.ref_lattices, nlat))
        t0 = time.perf_counter()
        ora.run_batch(ora.CHAR_POSITION, sub.lattices(), cores, label_group={0: 0, 1: 1}, inc_groups=[ora.INT_MAX],
                      del_groups=[1], **flags)
        dt = time.perf_counter() - t0
        cpu = {"value": sub.num_arcs / dt, "unit": "arcs/s", "cores": cores, "kind": "port",
               "sample": "first %d lattices, %.1f s on %d threads" % (len(sub), dt, cores)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.tool in (
            "frame_post", "segment", "position", "utterance", "best_path2", "position_post"):
        from oracle import ora
        ora.build()
        cores = os.cpu_count() or 1
        n = min(4 * args.ref_lattices, nlat)  # ~10-30 s of CPU work at full size
        if args.tool in ("position", "best_path2", "position_post"):
            n = min(n, 2 * cores)
        elif args.tool == "utterance":
            n = min(n, cores)
        sub = batch.slice(0, n)
        t0 = time.perf_counter()
        ora.run_batch(oracle_tool(ora, args.tool), sub.lattices(), cores, **flags)
        dt = time.perf_counter() - t0
        cpu = {"value": sub.num_arcs / dt, "unit": "arcs/s", "cores": cores, "kind": "port",
               "sample": "first %d lattices of the workload (%d arcs), one oracle run on %d host threads, %.1f s"
                         % (n, sub.num_arcs, cores, dt)}

    tools = None
    if rank == 0 and world == 1 and not args.no_tools and args.tool == "frame_post":
        if eng.h:
            eng.close()
        del batch, keep
        tools = bench_tools(klu, local, args, peak)

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "metric_note": METRIC_NOTE, "value": value, "unit": "arcs/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, nlat),
            "batch": {"lattices": st["lattices"], "states": states, "arcs": arcs, "levels": st["levels"],
                      "index_entries": entries, "gen_s": t_gen, "load_s": t_load, "total_arcs_all_ranks": total_arcs},
            "pack_ms": pack_total,
            "value_incl_pack": total_arcs / ((ms_per_step + pack_total) * 1e-3),
            "pack_note": "device time, once per batch, of the packer in klu_load plus the frame index "
                         "(the (frame, word) sort) built by the first frame-post run; `value` leaves it out, "
                         "`value_incl_pack` adds it to every step",
            "strong_scaling": strong,
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "tools": tools, "clocks": sampler.summary(), "numa": numa}))
    if eng.h:
        eng.close()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
