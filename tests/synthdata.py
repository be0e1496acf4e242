"""Deterministic synthetic indexes for tests and bench: genome from tools/synth.py, FM index
from the PRODUCT's own builder (unc_index_build, byte-identical to bwa), .uncl threshold line
from the committed fixture tests/golden/synth_uncl.json (made by the real reference)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import synth  # noqa: E402

CACHE = os.path.join(ROOT, "bench_data")


def get_index(name, cache=CACHE):
    """Returns (prefix, genome array).  Builds into `cache` (bench_data/ by default) on first use."""
    import ctypes as C
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "synth_uncl.json")))[name]
    os.makedirs(cache, exist_ok=True)
    prefix = os.path.join(cache, name)
    g = synth.genome(meta["size"], meta["seed"])
    if not all(os.path.exists(prefix + e) for e in (".bwt", ".sa", ".ann", ".amb", ".pac", ".uncl")):
        fa = prefix + ".fa"
        synth.write_fasta(fa, g)
        from uncalled_b200 import _native as N
        rc = N.lib().unc_index_build(fa.encode(), prefix.encode())
        if rc != 0:
            raise RuntimeError("unc_index_build failed: %d" % rc)
        open(prefix + ".uncl", "w").write(meta["uncl"])
    return prefix, g
