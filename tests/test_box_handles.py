"""Host-side behaviour of box ciphertext handles (spf_b200_box_ciphertext_*) that needs no GPU: argument validation,
the Python mirror's io checks, the single-context graph refusing a handle, and the C++ mirror compiling with -Werror."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fake_handle(kind: str, nbytes: int | None = None):
    """A BoxCiphertext object without a box behind it: enough for the host-side io checks."""
    import spf_b200

    h = spf_b200.BoxCiphertext.__new__(spf_b200.BoxCiphertext)
    h.kind, h.ptr = kind, 0x1000
    h.nbytes = spf_b200.io_bytes(kind) if nbytes is None else nbytes
    return h


def test_alloc_refuses_a_null_box_and_an_unknown_kind():
    import spf_b200

    l = spf_b200.lib()
    out = C.c_void_p(0x1234)
    assert l.spf_b200_box_ciphertext_alloc(None, spf_b200.OP["InputGlwe1"], C.byref(out)) == -1
    assert out.value is None and b"box is NULL" in l.spf_b200_box_last_error(None)
    for kind in (spf_b200.OP["OutputLwe0"], spf_b200.OP["CMux"], 0xFFFFFFFF):
        assert l.spf_b200_box_ciphertext_alloc(None, kind, C.byref(out)) == -1
        assert b"unknown kind" in l.spf_b200_box_last_error(None)


def test_write_read_free_refuse_what_is_not_a_live_handle():
    import spf_b200

    l = spf_b200.lib()
    buf = np.zeros(4096, np.uint64)
    assert l.spf_b200_box_ciphertext_write(None, buf.ctypes.data) == -1
    assert l.spf_b200_box_ciphertext_read(buf.ctypes.data, 0, buf.ctypes.data) == -1
    assert b"not a live handle" in l.spf_b200_box_last_error(None)
    l.spf_b200_box_ciphertext_free(None)
    l.spf_b200_box_ciphertext_free(buf.ctypes.data)  # not a handle: ignored
    assert not buf.any()


def test_check_io_takes_a_box_ciphertext_of_the_node_kind():
    import spf_b200
    from spf_b200 import OP, FheCircuit

    c = FheCircuit()
    for kind in ("Lwe0", "Lwe1", "Glwe1", "Ggsw1", "Glev1"):
        c._check_io(OP["Input" + kind], _fake_handle(kind))
        c._check_io(OP["Output" + kind], _fake_handle(kind))
    with pytest.raises(spf_b200.SpfError, match="holds a Lwe0"):
        c._check_io(OP["InputGlwe1"], _fake_handle("Lwe0"))
    with pytest.raises(spf_b200.SpfError, match="bytes"):
        c._check_io(OP["OutputGlwe1"], _fake_handle("Glwe1", 8))
    with pytest.raises(spf_b200.SpfError, match="takes no io"):
        c._check_io(OP["CMux"], _fake_handle("Glwe1"))
    n = c.add("InputGlwe1", io=_fake_handle("Glwe1"))
    assert c.nodes[n][3].kind == "Glwe1"


def test_compiled_graph_refuses_a_box_ciphertext():
    import spf_b200
    from spf_b200 import FheCircuit

    c = FheCircuit()
    c.add("OutputGlwe1", c.add("InputGlwe1", io=np.zeros(4096, np.uint64)), io=np.zeros(4096, np.uint64))
    g = spf_b200.CompiledGraph.__new__(spf_b200.CompiledGraph)
    g._keep = c
    with pytest.raises(spf_b200.SpfError, match="box graphs only"):
        g.set_io(0, _fake_handle("Glwe1"))


def test_cpp_box_ciphertext_mirror(tmp_path):
    """spf::BoxCiphertext of include/spf_b200.hpp compiles with -Werror next to BoxGraph, links, and a refused box
    creation still surfaces as spf::Error."""
    import shutil
    import subprocess

    import spf_b200

    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    src = tmp_path / "box_handle_smoke.cpp"
    src.write_text(r'''
#include <cstdio>
#include <vector>
#include "spf_b200.hpp"
int main() {
  const spf_params p = spf::default_128();
  try {
    spf::BoxEvaluation box(p, {}, {}, {}, {}, {});
    spf::BoxCiphertext mid(box, SPF_OP_INPUT_GLWE1);
    std::vector<std::uint64_t> host(spf_b200_len_glwe_l1(&p));
    mid.write(host.data());
    spf::FheCircuit c;
    c.output(SPF_OP_OUTPUT_GLWE1, c.input(SPF_OP_INPUT_GLWE1, host.data()), mid.handle());
    spf::BoxGraph g(box, c);
    g.set_io(1, mid.handle());
    g.run();
    mid.read(host.data(), 1);
  } catch (const spf::Error& e) {
    std::printf("box error %d: %s\n", e.code, e.what());
    return e.code == SPF_E_INVALID ? 0 : 1;
  }
  return 2;
}
''')
    lib_dir = os.path.dirname(spf_b200.LIB_PATH)
    exe = str(tmp_path / "box_handle_smoke")
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", lib_dir, "-l:" + os.path.basename(spf_b200.LIB_PATH), "-Wl,-rpath," + lib_dir])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert "box error -1" in out.stdout
