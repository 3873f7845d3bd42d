"""Write tests/golden/ref_calls.json: the reference's side of every test that takes the `ref` fixture
(tests/test_oracle_vs_ref.py, tests/test_graph_ext.py), recorded call by call -- see tests/refrecord.py.

    REF=<upstream source tree> python tests/golden/gen_golden_ref.py

With the upstream sources (or a built oracle/_ref/libref.so) the record is libref.so's own output.  Without them
it is written from the oracle's stand-in, which reproduces what the tests compare only where the oracle has been
pinned equal to libref.so on the same inputs: the committed record was written so, from the oracle that passed the
whole suite against libref.so (DESIGN.md section 2), and every later run with libref.so present checks it again.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tests import refrecord  # noqa: E402

env = dict(os.environ, CPROC_REF_RECORD=refrecord.RECORD)
rc = subprocess.call([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "not gpu",
                      os.path.join(ROOT, "tests", "test_oracle_vs_ref.py"), os.path.join(ROOT, "tests", "test_graph_ext.py")],
                     cwd=ROOT, env=env)
if rc:
    sys.exit("the tests failed while recording: %s not trusted" % refrecord.RECORD)
print("wrote", refrecord.RECORD, os.path.getsize(refrecord.RECORD), "bytes")
