"""ms per step of lattice-char-index-utterance next to lattice-char-index-position on the same batch
of synthetic c5 lattices (--nbest 100), a per-kernel profile of one utterance run, and the
KLU_CHAR_DEBUG lines of one run (DP tasks per depth, deepest frontier depth).

    python profiles/scripts/char_utterance_bench.py [--lattices 256] [--steps 5] [--out DIR]

Needs a CUDA device.  The card's name and power limit are printed with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lattices", type=int, default=256)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--nbest", type=int, default=100)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="directory for the debug log and the profile (default: a temp dir)")
    a = ap.parse_args()
    import __graft_entry__
    klu = __graft_entry__.load_package()
    out = a.out or tempfile.mkdtemp(prefix="char_utt_")
    os.makedirs(out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    batch = klu.synth_batch("c5", a.lattices, seed=a.seed)
    eng = klu.Engine(0)
    eng.load(batch)
    lg, inc, dele = klu.binding.char_groups([1], ())
    o, keep = klu.binding.make_opts(label_group=lg, inc_groups=inc, del_groups=dele, nbest=a.nbest)
    tools = {"char_position": klu.CHAR_POSITION, "char_utterance": klu.CHAR_UTTERANCE}
    res = {"card": card, "lattices": a.lattices, "states": int(batch.num_states), "nbest": a.nbest, "ms_per_step": {}}
    for name, t in tools.items():  # warm-up: module load, buffers grown to size
        eng.run_opts(t, o)
    for rep in range(2):  # alternate the tools
        for name, t in tools.items():
            eng.timer_start()
            for _ in range(a.steps):
                eng.run_opts(t, o)
            ms = eng.timer_stop() / a.steps
            res["ms_per_step"].setdefault(name, []).append(round(ms, 3))
    eng.profile(True)
    eng.run_opts(klu.CHAR_UTTERANCE, o)
    prof = eng.profile_json()
    eng.profile(False)
    with open(os.path.join(out, "char_utterance_profile.json"), "w") as f:
        json.dump(prof, f)
    # one run with KLU_CHAR_DEBUG: the library writes its lines to stderr (fd 2)
    log = os.path.join(out, "char_utterance_debug.txt")
    os.environ["KLU_CHAR_DEBUG"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    fd = os.open(log, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o644)
    os.dup2(fd, 2)
    try:
        eng.run_opts(klu.CHAR_UTTERANCE, o)
    finally:
        os.dup2(saved, 2)
        os.close(fd)
        del os.environ["KLU_CHAR_DEBUG"]
    lines = open(log).read().splitlines()
    tasks = [l for l in lines if "occurrence DP tasks" in l]
    depths = [int(l.split("depth ")[1].split(":")[0]) for l in lines if "candidates" in l]
    res["dp_tasks"] = sum(int(l.split(": ")[1].split()[0]) for l in tasks)
    res["dp_tasks_per_depth"] = [int(l.split(": ")[1].split()[0]) for l in tasks]
    res["deepest_depth"] = max(depths) if depths else 0
    res["profile"] = prof
    eng.close()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
