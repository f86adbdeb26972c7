"""CPU: per-layer chunk tables of a batch commit (mkhost_memfs_commit_layers with MKHOST_LAYER_TABLES) through the real
libmkhost packer against the CPU mock of the engine with its grouped-session calls
(tests/mock_engine/mock_mksnap_groups.cpp): the packer tags every file with its layer, and each layer's root / n_chunks /
n_unique must equal a separate commit of that layer.  Runs in a fresh process like tests/test_host_mock_engine_cpu.py,
and as an ordinary user (nothing is chowned).  With LD_PRELOAD of the sanitizer runtimes and a sanitized libmkhost
(the build line of tests/run_host_sanitized.sh) it reports any sanitizer finding as a failure."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def mock_so(tmp_path_factory):
    out = tmp_path_factory.mktemp("mock")
    obj, so = str(out / "mkoracle.o"), str(out / "libmock_mksnap.so")
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-c", os.path.join(ROOT, "oracle", "mkoracle.c"), "-o", obj])
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-Wall",
                           os.path.join(HERE, "mock_engine", "mock_mksnap_groups.cpp"), obj, "-o", so])
    return so


def test_batch_of_layers_with_layer_tables(mock_so, tmp_path):
    r = subprocess.run([sys.executable, "-m", "tests.mock_engine.layer_tables", mock_so, str(tmp_path)], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SCENARIO-OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]
    assert "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-6000:]  # tests/run_host_sanitized.sh
