"""Generates tests/golden/neuralnetapi_interface.json: the interface of the reference's NeuralNetAPI class
(engine/src/nn/neuralnetapi.h) that a back-end subclass builds on -- constructor and method signatures with their access,
virtual and pure flags, the data members with their types, the nn_api::Shape / NeuralNetDesign structs of
nn/neuralnetdesign.h, the Version typedefs and make_version() of version.h and the GamePhase typedef of state.h.  Only
types, names of members and these flags are recorded; no code.  interface_header() turns the record back into a
declaration-only header that tests/test_integration_stub.py compiles INTEGRATION.md's stub against.  Read from a CrazyAra
checkout, and checked by compiling the stub against both the real headers and the recorded interface:
    python tests/golden/gen_neuralnetapi_golden.py <CrazyAra checkout>"""
import json
import os
import re
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
GOLDEN = os.path.join(HERE, "neuralnetapi_interface.json")


def _strip_comments(src):
    return re.sub(r"//[^\n]*", "", re.sub(r"/\*.*?\*/", "", src, flags=re.S))


def _body(src, head):
    """Text between the braces of the first `head {` in src."""
    m = re.search(head + r"\s*\{", src)
    i, depth = m.end(), 1
    for j in range(i, len(src)):
        depth += {"{": 1, "}": -1}.get(src[j], 0)
        if depth == 0:
            return src[i:j]
    raise ValueError(head)


def _declarations(body):
    """(access, declaration) of a class body in order: inline function bodies dropped, access specifiers tracked."""
    out, cur, access, i = [], "", "private", 0
    while i < len(body):
        c = body[i]
        if c == "{":                      # an inline body ends the declaration
            depth = 1
            while depth:
                i += 1
                depth += {"{": 1, "}": -1}.get(body[i], 0)
            c = ";"
        if c == ";":
            d = " ".join(cur.split())
            while True:
                m = re.match(r"^(public|protected|private)\s*:\s*", d)
                if not m:
                    break
                access, d = m.group(1), d[m.end():]
            if d:
                out.append((access, d))
            cur = ""
        else:
            cur += c
            m = re.match(r"^\s*(public|protected|private)\s*:\s*$", cur)
            if m:
                access, cur = m.group(1), ""
        i += 1
    return out


def _param_types(params):
    params = params.strip()
    if not params or params == "void":
        return []
    return [re.match(r"^(.*?[\s&*])\w+$", p.strip()).group(1).strip() for p in params.split(",")]


def _members(body, name):
    members = []
    for access, d in _declarations(body):
        m = re.match(r"^(?P<spec>(?:(?:virtual|inline|static|explicit)\s+)*)(?P<ret>.*?)\s*\b(?P<name>~?\w+)\s*"
                     r"\((?P<params>[^)]*)\)\s*(?P<const>const)?\s*(?P<pure>=\s*0)?$", d)
        if m:
            members.append(dict(kind="ctor" if m["name"] == name else "method", access=access, name=m["name"],
                                ret=m["ret"], params=_param_types(m["params"]), virtual="virtual" in m["spec"],
                                const=bool(m["const"]), pure=bool(m["pure"])))
            continue
        m = re.match(r"^(?P<const>const\s+)?(?P<type>.+?)\s+(?P<name>\w+)(?P<arr>\[\d+\])?(?:\s*=.*)?$", d)
        members.append(dict(kind="field", access=access, name=m["name"], type=m["type"], const=bool(m["const"]),
                            array=m["arr"] or ""))
    return members


def record(checkout):
    src = os.path.join(checkout, "engine", "src")
    read = lambda p: _strip_comments(open(os.path.join(src, p)).read())  # noqa: E731
    api, design, version, state = read("nn/neuralnetapi.h"), read("nn/neuralnetdesign.h"), read("version.h"), read("state.h")
    typedefs = {}
    for text in (version, state):
        for t, n in re.findall(r"typedef\s+([\w:]+(?:\s+\w+)*)\s+(\w+)\s*;", text):
            if n in ("Version", "VersionType", "GamePhase"):
                typedefs[n] = t
    mv = re.search(r"inline\s+constexpr\s+(\w+)\s+make_version\(([^)]*)\)", version)
    return {"system_includes": sorted(set(re.findall(r"#include\s*<([^>]+)>", api + design))),
            "typedefs": typedefs,
            "make_version": dict(ret=mv.group(1), params=_param_types(mv.group(2))),
            "structs": {n: _members(_body(design, r"struct\s+" + n), n) for n in ("Shape", "NeuralNetDesign")},
            "NeuralNetAPI": _members(_body(api, r"class\s+NeuralNetAPI"), "NeuralNetAPI")}


def _member_decl(m):
    if m["kind"] == "field":
        # const members keep their initialised state without the reference's values
        return f"{'const ' if m['const'] else ''}{m['type']} {m['name']}{m['array']}{'{}' if m['const'] else ''};"
    params = ", ".join(m["params"])
    return (f"{'virtual ' if m['virtual'] else ''}{m['ret'] + ' ' if m['ret'] else ''}{m['name']}({params})"
            f"{' const' if m['const'] else ''}{' = 0' if m['pure'] else ''};")


def interface_header(rec):
    """A declaration-only neuralnetapi.h equivalent to the recorded interface."""
    lines = ["#pragma once", "#include <cstdint>"] + [f"#include <{h}>" for h in rec["system_includes"]]
    lines.append("using namespace std;")
    lines += [f"typedef {t} {n};" for n, t in rec["typedefs"].items()]
    mv = rec["make_version"]
    lines.append(f"inline constexpr {mv['ret']} make_version({', '.join(mv['params'])}) {{ return 0; }}")
    lines.append("namespace nn_api {")
    for name, members in rec["structs"].items():
        lines += [f"struct {name} {{"] + ["    " + _member_decl(m) for m in members] + ["};"]
    lines.append("}")
    lines.append("class NeuralNetAPI {")
    for m in rec["NeuralNetAPI"]:
        lines.append(f"{m['access']}:\n    {_member_decl(m)}")
    lines.append("};")
    return "\n".join(lines) + "\n"


def main(checkout):
    from tests.test_integration_stub import compile_stub
    rec = record(checkout)
    src = os.path.join(checkout, "engine", "src")
    with tempfile.TemporaryDirectory() as d:
        # the reference's headers reach its (absent) chess environment through stateobj.h; the repository's stand-ins for
        # the environment and for blaze (oracle/ref, see oracle/Makefile) let the header tree parse
        r = compile_stub(d, ["-DMODE_POMMERMAN", "-I" + os.path.join(ROOT, "oracle", "ref"), "-I" + src, "-I" + src + "/nn"])
        assert r.returncode == 0, "stub against the real headers:\n" + r.stderr[-3000:]
        with open(os.path.join(d, "neuralnetapi.h"), "w") as f:
            f.write(interface_header(rec))
        r = compile_stub(d, ["-I" + d])
        assert r.returncode == 0, "stub against the recorded interface:\n" + r.stderr[-3000:]
    with open(GOLDEN, "w") as f:
        json.dump(rec, f, indent=1)
    print("wrote", GOLDEN, len(rec["NeuralNetAPI"]), "NeuralNetAPI members")


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    main(sys.argv[1])
