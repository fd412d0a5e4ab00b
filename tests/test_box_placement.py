"""Host-side behaviour of box graph placement (spf_b200_box_graph_build_on) that needs no GPU: the Python checks of
`ranks` that run before any C call, the NULL arguments of the C entry points, and the C++ overloads compiling with
-Werror."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _circuit():
    from spf_b200 import FheCircuit

    c = FheCircuit()
    c.add("OutputGlwe1", c.add("Not", c.add("InputGlwe1", io=np.zeros(4096, np.uint64))), io=np.zeros(4096, np.uint64))
    return c


def test_single_context_processor_refuses_ranks():
    import spf_b200

    ev = spf_b200.Evaluation.__new__(spf_b200.Evaluation)  # no context behind it: the check comes first
    proc = spf_b200.CircuitProcessor(ev)
    for ranks in ([0], [], (1, 0)):
        with pytest.raises(spf_b200.SpfError) as e:
            proc.compile(_circuit(), ranks=ranks)
        assert e.value.code == -1 and "BoxEvaluation" in str(e.value)
    with pytest.raises(spf_b200.SpfError) as e:
        proc.spawn_graph(_circuit(), ranks=[0])
    assert e.value.code == -1
    errs = []
    assert proc.spawn_graph(_circuit(), on_completion=errs.append, ranks=[0]) is None
    assert len(errs) == 1 and isinstance(errs[0], spf_b200.SpfError) and errs[0].code == -1


def test_box_graph_ranks_must_be_rank_numbers():
    import spf_b200

    box = spf_b200.BoxEvaluation.__new__(spf_b200.BoxEvaluation)  # no box behind it: the check comes first
    for ranks in (["0"], [0.0], [None], 1, [2 ** 31], [-2 ** 31 - 1]):
        with pytest.raises(spf_b200.SpfError) as e:
            spf_b200.BoxGraph(box, _circuit(), ranks=ranks)
        assert e.value.code == -1 and "ranks" in str(e.value)
    with pytest.raises(spf_b200.SpfError):
        spf_b200.CircuitProcessor(box).compile(_circuit(), ranks=[0.5])


def test_build_on_and_ranks_refuse_null():
    import spf_b200

    l = spf_b200.lib()
    c = _circuit()
    out = C.c_void_p(0x1234)
    ranks = (C.c_int * 1)(0)
    assert l.spf_b200_box_graph_build_on(None, c._pack(), len(c.nodes), ranks, 1, C.byref(out)) == -1
    assert l.spf_b200_box_graph_ranks(None, None) == -1
    assert l.spf_b200_box_graph_ranks(None, ranks) == -1


def test_cpp_placement_overloads(tmp_path):
    """spf::BoxGraph(box, circuit, ranks), BoxCircuitProcessor::compile(circuit, ranks) and BoxGraph::ranks() compile
    with -Werror and link; a refused box creation still surfaces as spf::Error."""
    import shutil
    import subprocess

    import spf_b200

    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    src = tmp_path / "box_place_smoke.cpp"
    src.write_text(r'''
#include <cstdio>
#include <vector>
#include "spf_b200.hpp"
int main() {
  const spf_params p = spf::default_128();
  try {
    spf::BoxEvaluation box(p, {}, {}, {}, {}, {});
    std::vector<std::uint64_t> host(2 * spf_b200_len_glwe_l1(&p));
    spf::FheCircuit c;
    c.output(SPF_OP_OUTPUT_GLWE1, c.add(SPF_OP_NOT, c.input(SPF_OP_INPUT_GLWE1, host.data())), host.data() + host.size() / 2);
    spf::BoxGraph g(box, c, std::vector<int>{1});
    spf::BoxCircuitProcessor proc(box);
    spf::BoxGraph h = proc.compile(c, {1, 0});
    const std::vector<int> r = g.ranks();
    h.spawn({&g}, nullptr, nullptr);
    h.wait();
    return r.size() == 1 ? 3 : 4;
  } catch (const spf::Error& e) {
    std::printf("box error %d: %s\n", e.code, e.what());
    return e.code == SPF_E_INVALID ? 0 : 1;
  }
  return 2;
}
''')
    lib_dir = os.path.dirname(spf_b200.LIB_PATH)
    exe = str(tmp_path / "box_place_smoke")
    subprocess.check_call([cxx, "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src),
                           "-o", exe, "-L", lib_dir, "-l:" + os.path.basename(spf_b200.LIB_PATH), "-Wl,-rpath," + lib_dir])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, (out.returncode, out.stdout, out.stderr)
    assert "box error -1" in out.stdout
