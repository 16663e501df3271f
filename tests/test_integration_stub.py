"""INTEGRATION.md shows the reference-side binding a maintainer would add: `class B200API : public NeuralNetAPI` over the
C-ABI.  This test extracts that C++ block and compiles it against the interface of the reference's REAL NeuralNetAPI
(nn/neuralnetapi.h: constructor, virtual hooks and their access, data members and the NeuralNetDesign struct, recorded
from the reference's headers in tests/golden/neuralnetapi_interface.json by gen_neuralnetapi_golden.py, which also
compiles the stub against the headers themselves), so the stub cannot drift from the interface it claims to implement."""
import json
import os
import re
import subprocess

from tests.golden.gen_neuralnetapi_golden import GOLDEN, interface_header

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def compile_stub(work_dir, include_flags):
    """g++ -fsyntax-only of INTEGRATION.md's B200API block with the given -I / -D flags; the stub must implement every
    pure virtual (an instantiable back-end)."""
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    blocks = re.findall(r"```cpp\n(.*?)```", md, re.S)
    stub = next(b for b in blocks if "class B200API" in b)
    src = os.path.join(work_dir, "b200api.cpp")
    with open(src, "w") as f:
        f.write("#define BACKEND_B200 1\n#include <type_traits>\n" + stub +
                "\nstatic_assert(!std::is_abstract<B200API>::value, \"B200API leaves a pure virtual open\");"
                "\nint main() { return sizeof(B200API) > 0 ? 0 : 1; }\n")
    cmd = ["g++", "-std=c++17", "-fsyntax-only", "-w"] + include_flags + ["-I" + os.path.join(ROOT, "include"), src]
    return subprocess.run(cmd, capture_output=True, text=True)


def test_b200api_stub_compiles_against_the_reference_header(tmp_path):
    with open(GOLDEN) as f:
        rec = json.load(f)
    (tmp_path / "neuralnetapi.h").write_text(interface_header(rec))
    r = compile_stub(str(tmp_path), ["-I" + str(tmp_path)])
    assert r.returncode == 0, r.stderr[-3000:]
