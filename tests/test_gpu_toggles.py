"""The run-time switches of the library (read once per process) must not change any result: a parity test
with > 1 M queries (several pipeline chunks, query sorting active) is re-run in subprocesses with the
alternative code paths selected."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOGGLES = [
    {"GDX_VERIFY": "0", "GDX_SORT_QUERIES": "0", "GDX_DENSE_SA": "0", "GDX_SEED_TABLE": "0", "GDX_CHUNK_FIRST_MB": "1", "GDX_CHUNK_MAX_MB": "2",
     "GDX_CHUNK_TAIL_MB": "1"},
    {"GDX_FORCE_WIDE": "1", "GDX_VERIFY_MIN": "2", "GDX_CHUNK_MAX_MB": "256"},
    # every batch, however small, takes the host packer + packed kernel + staged uint32 results
    {"GDX_PACK_MIN_BYTES": "0", "GDX_STAGE_MIN_BYTES": "0", "GDX_CHUNK_FIRST_MB": "1", "GDX_CHUNK_MAX_MB": "1"},
    {"GDX_PACK_MIN_BYTES": "0", "GDX_STAGE_MIN_BYTES": "0", "GDX_VERIFY": "0", "GDX_SEED_TABLE": "0", "GDX_HOST_THREADS": "3",
     "GDX_PACK_SCALAR": "1"},
    # round-1 transfer paths: IO bytes and uint64 results over PCIe
    {"GDX_PACK_QUERIES": "0", "GDX_NARROW_RESULTS": "0"},
]


@pytest.mark.parametrize("env", TOGGLES, ids=["lfonly-nosort-smallchunks", "wide-verifymin2", "pack-everything",
                              "pack-everything-lfonly-scalar", "no-pack-no-narrow"])
def test_parity_under_toggles(env):
    e = dict(os.environ)
    e.update(env)
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_parity.py"), "-m", "gpu",
                          "-q", "-x", "-p", "no:cacheprovider", "-k",
                          "chunking or verification_shortcut or cursor_shortcut or many_hits or dense_suffix or seed_table "
                          "or kat or invalid or unsearchable"],
                         env=e, capture_output=True, text=True, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
