"""Runs the C++ contract test of the drop-in VectorIndex subclass for the binary index types
(dingo-store_b200/host/test_plugin_binary.cc)."""
import os
import subprocess

import pytest

import b200vs
from gpu_util import require_gpu

pytestmark = pytest.mark.gpu


def test_cpp_binary_plugin_contract():
    require_gpu()
    exe = os.path.join(b200vs.PKG_ROOT, "host", "test_plugin_binary")
    assert os.path.exists(exe), "build it with: make -C dingo-store_b200/host"
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    print(r.stdout[-3000:])
    assert r.returncode == 0 and "BINARY PLUGIN TESTS OK" in r.stdout, r.stdout[-3000:] + r.stderr[-1000:]
