"""The tight pin of the oracle: `python oracle/ref_harness.py check` imports the REFERENCE's own modules (behind the harness
shims) and compares the oracle with them in the same process — servers bit-identical, per-sample tensors and renders at 1e-4
(>= 97 % of entries, 30x tolerance on the rest), background bit-identical, pose-server gradients.  It needs the reference's
source tree (oracle.ref_harness.REF), which is not part of this repository: where it exists this test runs the harness (in a
fresh interpreter: the shims patch torch.Tensor.cuda) and requires "ORACLE == REFERENCE"; elsewhere it skips, and
tests/test_cpu_oracle.py (oracle vs the committed reference-generated goldens) is the self-contained check."""
import os
import subprocess
import sys

import pytest

from oracle.ref_harness import REF

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not os.path.isdir(REF), reason="the reference implementation's source tree is not present")
def test_oracle_equals_reference_modules():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_harness.py"), "check"], capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-3000:]
    assert r.returncode == 0, tail + r.stderr[-2000:]
    assert "ORACLE == REFERENCE" in r.stdout and "MISMATCH" not in r.stdout, tail
