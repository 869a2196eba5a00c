"""B200-native lattice forward-backward / posterior-indexing engine.

Drop-in for the hot path of jpuigcerver/kaldi-lattice-utils (see DESIGN.md).  The
directory name carries a hyphen (it mirrors the reference's repository name), so
import it through `__graft_entry__.load_package()` / importlib, e.g.

    import importlib.util, sys
    spec = importlib.util.spec_from_file_location(
        "klu_b200", "kaldi-lattice-utils_b200/__init__.py",
        submodule_search_locations=["kaldi-lattice-utils_b200"])
    klu = importlib.util.module_from_spec(spec); sys.modules["klu_b200"] = klu
    spec.loader.exec_module(klu)
"""
from . import binding, lattice, shard  # noqa: F401
from .binding import (BEST_PATH2, CHAR_POSITION, CHAR_SEGMENT, CHAR_UTTERANCE, FRAME_POST, LENGTH_DIST, FWD_BWD, POSITION, POSITION_POST, PRUNE_ARCS, PRUNE_DYN_BEAM,  # noqa: F401
                      SEGMENT,
                      UTTERANCE, Engine, KluError)
from .lattice import (Lattice, LatticeBatch, format_tuples, kaldi_float, make_lattice, read_text_ark,  # noqa: F401
                      synth_batch, topsort)
from .shard import partition_by_arcs, run_sharded  # noqa: F401,E402
