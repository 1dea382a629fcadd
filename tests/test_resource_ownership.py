"""GPU tier: a create call that fails after it has allocated releases what it allocated."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# W = 400, S = 4000 passes every parameter check, but the fused kernel's shared-memory layout then needs 295 168 B, more
# than a block may use. MfccCuda finds that out after it has created its stream, its two pinned PCM staging buffers
# (about 20 MB each at an input buffer of 10 000 000 samples) and the FFT twiddle tables. The creations run in a child
# process, so that whatever they might leak stays out of the test process. Pinned pages count in VmRSS (as RssShmem):
# when the failed creations leaked them, VmRSS grew by about 760 MB on a B200 host.
CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import afe_loader
afe = afe_loader.load()

def status_kb():
    with open("/proc/self/status") as f:
        return {k: int(v.split()[0]) for k, v in (l.split(":", 1) for l in f) if k.startswith(("Vm", "Rss"))}

afe.MfccCuda(afe.make_params()).close()  # the CUDA context and the allocators exist before the first reading
before = status_kb()
errors = []
for _ in range(20):
    try:
        afe.MfccCuda(afe.make_params(window_size=400, shift=4000, input_buffer_size=10_000_000)).close()
        errors.append(None)
    except afe.AfeError as e:
        errors.append(str(e))
print(json.dumps({"before": before, "after": status_kb(), "errors": errors}))
"""


def test_failed_mfcc_create_releases_pinned_buffers():
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert len(res["errors"]) == 20 and all(m and "shared-memory budget" in m for m in res["errors"]), res["errors"]
    grown_mb = (res["after"]["VmRSS"] - res["before"]["VmRSS"]) / 1024
    assert grown_mb <= 100, f"the resident set grew by {grown_mb:.0f} MB over 20 failed creations: {res}"
