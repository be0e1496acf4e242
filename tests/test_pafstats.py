"""uncalled_b200/pafstats.py against the reference's own uncalled/pafstats.py: character for character against what that
script printed (stored), and the printed numbers pinned by hand."""
import io
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from uncalled_b200 import pafstats as PS  # noqa: E402

QRY = """r1\t450\t10\t400\t+\tchr\t100000\t5000\t5390\t40\t391\t255\tch:i:1\tst:i:0\tmt:f:12.500000
r2\t450\t0\t300\t-\tchr\t100000\t90000\t90300\t30\t301\t255\tch:i:2\tst:i:0\tmt:f:20.000000
r3\t450\t*\t*\t*\t*\t*\t*\t*\t*\t*\t255\tch:i:3\tst:i:0
r4\t450\t20\t200\t+\tchr\t100000\t700\t880\t25\t181\t255\tch:i:4\tst:i:0\tmt:f:5.000000
r5\t450\t*\t*\t*\t*\t*\t*\t*\t*\t*\t255\tch:i:5\tst:i:0
"""
REF = """r1\t450\t0\t450\t+\tchr\t100000\t4990\t5440\t400\t451\t60
r2\t450\t0\t450\t+\tchr\t100000\t20000\t20450\t400\t451\t60
r3\t450\t0\t450\t+\tchr\t100000\t100\t550\t400\t451\t60
r5\t450\t*\t*\t*\t*\t*\t*\t*\t*\t*\t255
"""


def test_summary_and_comparison(tmp_path):
    q, r = tmp_path / "q.paf", tmp_path / "r.paf"
    q.write_text(QRY)
    r.write_text(REF)
    buf = io.StringIO()
    s = PS.run(str(q), str(r), out=buf)
    assert (s["reads"], s["mapped"]) == (5, 3)
    assert s["vs_reference"] == {"tp": 1, "fp": 1, "na": 1, "tn": 1, "fn": 1, "n": 5}
    assert "T  20.00 20.00" in buf.getvalue() and "F  20.00 20.00" in buf.getvalue() and "NA: 20.00" in buf.getvalue()


def test_same_output_as_the_reference_script(tmp_path):
    """What the reference's uncalled/pafstats.py prints for the same two files, stored in tests/golden/reference_checks.json
    (tools/make_reference_checks_golden.py)."""
    import orclib
    q, r = tmp_path / "q.paf", tmp_path / "r.paf"
    q.write_text(QRY)
    r.write_text(REF)
    buf = io.StringIO()
    PS.run(str(q), str(r), out=buf)
    assert buf.getvalue() == orclib.reference_checks("pafstats")["stdout"]
