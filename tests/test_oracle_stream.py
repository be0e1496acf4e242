"""The oracle's restatement of the STREAMING path (EventProfiler, streaming Normalizer, chunked
process_chunk / map_chunk) against (a) committed results of the reference's own streaming path
(tests/golden/stream_golden.json, made by tools/make_stream_golden.py from oracle/_ref) and
(b) the same on fresh synthetic reads (tests/golden/reference_checks.json)."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import make_stream_golden as msg  # noqa: E402

GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "stream_golden.json")))


def _chunk_len(chunk_time):
    return int(np.float32(chunk_time) * np.float32(4000.0))      # ReadBuffer::PRMS.chunk_len(): u16(chunk_time * sample_rate)


@pytest.mark.parametrize("which", ["example", "g200k"])
def test_stream_port_matches_reference_golden(which):
    import orclib
    prefix, sigs = msg.signals(which)
    O = orclib.Oracle(prefix)
    for row in GOLD[which]:
        rec, nu, en = O.stream_read(sigs[row["read"]], _chunk_len(row["chunk_time"]), row["max_chunks"])
        assert list(orclib.paf_tuple(rec)) == row["paf"] and nu == row["chunks"] and en == row["ended"], row


def test_example_read_streams_like_uncalled_map_ord():
    """SURVEY 8(c): `uncalled_map_ord` on the example read prints ... 67 41 67 - ... 10000 6948 6977 29 30 255."""
    row = [r for r in GOLD["example"] if r["read"] == 0 and r["chunk_time"] == 1.0][0]
    p = row["paf"]
    assert p[0] == 1 and p[1] == 0 and p[6:11] == [67, 41, 67, 6948, 6977] and p[5] == 29


def test_stream_port_matches_ref_library_live():
    """bit-for-bit against the reference's own streaming Mapper (oracle/_ref) on fresh reads; its records are stored in
    tests/golden/reference_checks.json (tools/make_reference_checks_golden.py)."""
    import orclib
    import synth
    import synthdata
    rows = orclib.reference_checks("stream")["rows"]
    assert len(rows) == 30
    prefix, g = synthdata.get_index("g200k")
    O = orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 10, 9000, seed=77, frac_random=0.3)
    for row in rows:
        rec, nu, en = O.stream_read(np.ascontiguousarray(sig[row["read"]], np.float32), _chunk_len(row["chunk_time"]), row["max_chunks"])
        assert (list(orclib.paf_tuple(rec)), nu, en) == (row["paf"], row["chunks"], row["ended"]), row
