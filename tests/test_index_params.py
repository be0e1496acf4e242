"""`uncalled index` after the BWA build (SURVEY 8(f) rank 3): self_align + the parameter search.

Pins, in this order:
  * the oracle's self_align against digests of the reference's own C++ self_align
    (tests/golden/self_align_golden.json, tools/make_selfalign_golden.py and tests/golden/reference_checks.json);
  * uncalled_b200.index_params against (a) the `.uncl` file the reference SHIPS with its example index,
    (b) lines written by the real `uncalled index` for seeded genomes (tests/golden/synth_uncl.json) and
    (c) multi-preset files written by the reference's own IndexParameterizer
    (tests/golden/uncl_presets.json, tools/make_uncl_presets_golden.py) -- character for character."""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
from uncalled_b200 import index_params as IP  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
SA_GOLD = json.load(open(os.path.join(GOLD, "self_align_golden.json")))
PRESETS = json.load(open(os.path.join(GOLD, "uncl_presets.json")))
SYNTH = json.load(open(os.path.join(GOLD, "synth_uncl.json")))

_prefix = {}


def prefix_of(which):
    import orclib
    import synthdata
    if which not in _prefix:
        _prefix[which] = (orclib.materialise_example_index(tempfile.mkdtemp()) if which == "example"
                          else synthdata.get_index(which)[0])
    return _prefix[which]


_paths = {}


def paths_of(which, sample_dist):
    import orclib
    if (which, sample_dist) not in _paths:
        _paths[which, sample_dist] = orclib.self_align(prefix_of(which), sample_dist)
    return _paths[which, sample_dist]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, "<u8").tobytes()).hexdigest()


@pytest.mark.parametrize("row", SA_GOLD, ids=lambda r: "%s-%d" % (r["index"], r["sample_dist"]))
def test_oracle_self_align_matches_reference_digest(row):
    off, val = paths_of(row["index"], row["sample_dist"])
    assert (len(off) - 1, len(val)) == (row["n_paths"], row["n_values"])
    assert [[int(v) for v in val[int(off[i]):int(off[i + 1])]] for i in range(3)] == row["head"]
    assert sha(off) == row["offsets_sha256"] and sha(val) == row["values_sha256"]


def test_oracle_self_align_matches_ref_library_live():
    """Against the reference's own self_align (oracle/_ref) on the 200 kb index at three sampling distances; its
    digests are stored in tests/golden/reference_checks.json (tools/make_reference_checks_golden.py)."""
    import orclib
    from make_reference_checks_golden import sa_digest
    gold = orclib.reference_checks("self_align_g200k")
    for sd in (1, 7, 250):
        assert sa_digest(*paths_of("g200k", sd)) == gold[str(sd)], sd


def test_sample_distance_rules():
    """uncalled/index.py:76-82 with the `uncalled index` defaults (uncalled/args.py:87-137)."""
    assert IP.sample_distance(10000) == 1                   # ceil(10000 / 50000)
    assert IP.sample_distance(200000) == 4
    assert IP.sample_distance(4700000) == 94
    assert IP.sample_distance(5000000) == 100               # exactly min_samples at the maximum distance
    assert IP.sample_distance(50000000) == 100
    assert IP.sample_distance(230000000) == 230             # floor(ref_len / max_samples)
    assert IP.sample_distance(1000000, max_sample_dist=50, min_samples=20000) == 50


def test_uncl_of_shipped_example_index_is_the_shipped_file():
    """The reference ships example/example_ref.uncl next to its example index: regenerate it."""
    prefix = prefix_of("example")
    assert IP.reference_length(prefix) == 10000
    off, val = paths_of("example", IP.sample_distance(10000))
    assert IP.uncl_text(off, val) == open(prefix + ".uncl").read()


@pytest.mark.parametrize("which", ["g200k", "g1m"])
def test_uncl_matches_real_uncalled_index_run(which):
    prefix = prefix_of(which)
    off, val = paths_of(which, IP.sample_distance(IP.reference_length(prefix)))
    assert IP.uncl_text(off, val) == SYNTH[which]["uncl"]


@pytest.mark.parametrize("row", PRESETS, ids=lambda r: r["index"] + "-" + "-".join(sorted(r["opts"])))
def test_presets_match_reference_parameterizer(row):
    prefix = prefix_of(row["index"])
    o = dict(IP.DEFAULTS, **row["opts"])
    sd = IP.sample_distance(IP.reference_length(prefix), o["max_sample_dist"], o["min_samples"], o["max_samples"])
    off, val = paths_of(row["index"], sd)
    assert IP.uncl_text(off, val, probs=row["probs"], speeds=row["speeds"], **row["opts"]) == row["uncl"]


def test_unparsable_targets_are_skipped_like_the_cli():
    off, val = paths_of("example", 1)
    assert IP.uncl_text(off, val, probs="x,0.5", speeds=["-"]).splitlines()[1].startswith("prob_0.5\t")
    assert len(IP.uncl_text(off, val, probs="x", speeds="y").splitlines()) == 1


def test_index_cmd_end_to_end_with_the_emulated_device(tmp_path):
    """`uncalled index` from a FASTA alone: the product's FM-index builder, the device self-alignment source under
    the CPU emulator (injected in place of the GPU call) and the parameter search reproduce the index files AND the
    .uncl file that the reference ships for its example, and a multi-preset file of the reference's parameterizer."""
    import emulib
    import orclib
    from uncalled_b200 import index as UI
    os.makedirs(tmp_path / "src")
    src = orclib.materialise_example_index(str(tmp_path / "src"))
    fa = str(tmp_path / "example_ref.fa")
    open(fa, "wb").write(open(src + ".fa", "rb").read())
    row = PRESETS[0]
    assert row["index"] == "example" and not row["opts"]
    UI.index_cmd(fa, probs=row["probs"], speeds=row["speeds"], self_align_fn=emulib.self_align)
    for ext in (".bwt", ".sa", ".ann", ".amb", ".pac"):
        assert open(fa + ext, "rb").read() == open(src + ext, "rb").read(), ext
    assert open(fa + ".uncl").read() == row["uncl"]
    assert row["uncl"].splitlines()[0] + "\n" == open(src + ".uncl").read()          # its first line is the shipped file
    os.remove(fa + ".uncl")
    UI.index_cmd(fa, self_align_fn=emulib.self_align)                                 # BWA files are reused now
    assert open(fa + ".uncl").read() == open(src + ".uncl").read()
