"""Host-side behaviour of the box API (spf_b200_box_*) that needs no GPU: argument validation before any device is
touched, a loud failure without a device, the batch split, and the C++ mirror compiling with -Werror."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def _create(l, p, devices, n, lens=None):
    dummy = np.zeros(8, dtype=np.uint64)
    lens = lens or [8, 8, 8, 8]
    h = C.c_void_p()
    devs = None if devices is None else (C.c_int * max(len(devices), 1))(*devices)
    rc = l.spf_b200_box_create(C.byref(p), dummy.ctypes.data, lens[0], dummy.ctypes.data, lens[1], dummy.ctypes.data,
                               lens[2], dummy.ctypes.data, lens[3], devs, n, C.byref(h))
    return rc, h


def test_box_create_validates_arguments_before_any_device():
    """n = 0, n > 8 (a rank has at most 7 peers) and NULL devices are refused with SPF_E_INVALID -- not SPF_E_CUDA,
    which is what touching a device first would give here."""
    import spf_b200

    l = spf_b200.lib()
    p = spf_b200.default_128()
    for devices, n, what in (([0], 0, b"1..8"), ([0] * 9, 9, b"1..8"), (None, 2, b"devices is NULL")):
        rc, h = _create(l, p, devices, n)
        assert rc == -1 and not h.value, (n, rc)
        assert what in l.spf_b200_box_last_error(None)
    rc, _ = _create(l, p, [0, 0], 2)
    assert rc == -1 and b"key length" in l.spf_b200_box_last_error(None)
    buf = np.zeros(16, dtype=np.uint8)
    h = C.c_void_p()
    rc = l.spf_b200_box_create_from_serialized(C.byref(p), buf.ctypes.data, buf.size, None, 1, C.byref(h))
    assert rc == -1 and b"devices is NULL" in l.spf_b200_box_last_error(None)


@pytest.mark.skipif(_has_gpu(), reason="checks the behaviour without a CUDA device")
def test_box_create_fails_loudly_without_gpu():
    import spf_b200

    l = spf_b200.lib()
    p = spf_b200.default_128()
    lens = [l.spf_b200_len_bsk(C.byref(p)), l.spf_b200_len_ksk(C.byref(p)), l.spf_b200_len_ssk(C.byref(p)),
            l.spf_b200_len_ak(C.byref(p))]
    rc, h = _create(l, p, [0, 0], 2, lens)
    assert rc == -3 and not h.value
    assert b"no CPU fallback" in l.spf_b200_box_last_error(None)


def test_box_split_matches_multi_shard():
    import spf_b200
    from spf_b200 import multi

    for n in range(1, 9):
        for batch in (0, 1, 7, 8, 300, 301, 4096 * n + 5):
            got = [spf_b200.box_shard(batch, n, r) for r in range(n)]
            assert got == [multi.shard(batch, n, r) for r in range(n)], (batch, n)


def test_box_ops_refuse_a_null_box():
    import spf_b200

    l = spf_b200.lib()
    assert l.spf_b200_box_circuit_bootstrap(None, None, None, 1) == -1
    assert l.spf_b200_box_graph_run(None) == -1
    assert l.spf_b200_box_size(None) == 0 and l.spf_b200_box_context(None, 0) is None


def test_cpp_box_mirror(tmp_path):
    """spf::BoxEvaluation / BoxGraph / BoxCircuitProcessor of include/spf_b200.hpp compile with -Werror, link, and turn a
    refused creation into spf::Error."""
    import shutil
    import subprocess

    import spf_b200

    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    src = tmp_path / "box_smoke.cpp"
    src.write_text(r'''
#include <cstdio>
#include "spf_b200.hpp"
int main() {
  const spf_params p = spf::default_128();
  try {
    spf::BoxEvaluation box(p, {}, {}, {}, {}, {});
    spf::BoxCircuitProcessor proc(box);
    spf::FheCircuit c;
    proc.compile(c).run();
  } catch (const spf::Error& e) {
    std::printf("box error %d: %s\n", e.code, e.what());
    return e.code == SPF_E_INVALID ? 0 : 1;
  }
  return 2;
}
''')
    lib_dir = os.path.dirname(spf_b200.LIB_PATH)
    exe = str(tmp_path / "box_smoke")
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", lib_dir, "-l:" + os.path.basename(spf_b200.LIB_PATH), "-Wl,-rpath," + lib_dir])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert "box error -1" in out.stdout
