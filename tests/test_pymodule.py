"""The `_uncalled` extension module (uncalled_b200/csrc/pyuncalled.cpp): the name under which the reference's Python
package loads its C++ core (reference uncalled/__init__.py:1, src/pybinder.cpp:14-91).  CPU tier: it builds, exports
what `scripts/uncalled` and `uncalled/args.py` use, and formats PAF lines as the reference does.  GPU tier: MapPool maps
the example fast5 to the reference's golden PAF line."""
import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "uncalled_b200")
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "example_paf.json")))


def _module():
    sys.path.insert(0, ROOT)
    import uncalled_b200
    uncalled_b200.build()
    import uncalled_b200._native as N
    N.build_pymodule()
    if PKG not in sys.path:
        sys.path.insert(0, PKG)
    import _uncalled
    return _uncalled


def test_module_exports_the_names_the_reference_cli_uses():
    m = _module()
    for name in ("Conf", "Paf", "MapPool", "RealtimePool", "Chunk", "BwaIndex", "ClientSim", "self_align"):
        assert hasattr(m, name), name
    c = m.Conf()
    assert (c.max_events, c.idx_preset, c.threads, c.num_channels, c.max_chunks, c.chunk_time) == (30000, "default", 1, 512, 1000000, 1.0)
    assert m.Conf.read_list.__doc__ and m.Conf.max_reads.__doc__ and m.Conf.host.__doc__      # uncalled/args.py:223-260
    c.bwa_prefix, c.max_chunks = "x", 3
    assert (c.bwa_prefix, c.max_chunks) == ("x", 3)
    assert int(m.RealtimePool.DEPLETE) == 0 and int(m.RealtimePool.ENRICH) == 1 and int(m.RealtimePool.ODD) == 2
    assert int(m.Paf.ENDED) == 10 and int(m.Paf.KEEP) == 11
    # the DTW classes and presets of src/pybinder.cpp:75-91 (DTW_RAW_QSUB / _RSUB are bound to the EVENT presets there)
    for name in ("DTWr94p", "DTWr94d", "DTWParams", "DTW_EVENT_GLOB", "DTW_RAW_GLOB", "DTW_EVENT_QSUB", "DTW_EVENT_RSUB", "DTW_RAW_QSUB", "DTW_RAW_RSUB"):
        assert hasattr(m, name), name
    assert (m.DTW_EVENT_GLOB.dw, m.DTW_EVENT_GLOB.hw, m.DTW_EVENT_GLOB.vw) == (2, 1, 100)
    assert (m.DTW_RAW_GLOB.dw, m.DTW_RAW_GLOB.vw, m.DTW_RAW_QSUB.dw, m.DTW_RAW_RSUB.vw) == (10, 1000, 2, 100)


def test_paf_line_formatting_matches_the_golden_line():
    m = _module()
    f = GOLD["default"]["line"].split("\t")
    p = m.Paf(f[0], int(f[12].split(":")[2]), int(f[13].split(":")[2]))
    assert p.line().split("\t")[2:12] == ["*"] * 9 + ["255"]
    from uncalled_b200.api import Paf as PyPaf
    q = PyPaf(f[0], int(f[12].split(":")[2]), int(f[13].split(":")[2]))
    assert p.line() == q.line()
    p.set_float(m.Paf.MAP_TIME, 12.5)
    p.set_int(m.Paf.DELAY, 3)
    assert p.line().endswith("\tdl:i:3\tmt:f:12.500000")


@pytest.mark.gpu
def test_map_pool_maps_the_example_fast5_to_the_golden_line(tmp_path):
    """What `scripts/uncalled map -t 1 example_ref example.fast5` does (scripts/uncalled:127-167), on the pybind11 module."""
    m = _module()
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orclib
    prefix = orclib.materialise_example_index(str(tmp_path))
    for key, mod in (("default", {}), ("max_chunks_1", {"max_chunks": 1}), ("max_events_100", {"max_events": 100})):
        if key not in GOLD:
            continue
        conf = m.Conf()
        conf.bwa_prefix = prefix
        for k, v in mod.items():
            setattr(conf, k, v)
        pool = m.MapPool(conf)
        pool.add_fast5(os.path.join(ROOT, "tests", "golden", "fast5", "example_single.fast5"))
        out = []
        while pool.running():
            out += pool.update()
        pool.stop()
        assert len(out) == 1
        assert out[0].line().split("\t")[:14] == GOLD[key]["line"].split("\t")[:14], key
