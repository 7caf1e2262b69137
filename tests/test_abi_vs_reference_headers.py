"""The boundary, checked against the REFERENCE's own headers by the C compiler: tests/abi/abi_probe.c compiled against
include/aresdb_b200/*.h must print what it printed when compiled against the reference's query/time_series_aggregate.h +
cgoutils/memory.h (stored in tests/golden/abi_layout_reference.txt) — every struct size, field offset and enum value must
agree —, every function the reference's headers declare must have the same prototype in include/aresdb_b200/*.h, and the
probe linked against aresdb_b200/lib must bind to the B200 libraries and run."""
import hashlib
import re
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
REFERENCE_LAYOUT = ROOT / "tests" / "golden" / "abi_layout_reference.txt"
# "<function> <sha256 of its prototype>" for every function the reference's query/time_series_aggregate.h and
# cgoutils/memory.h declare, as prototype_digests() computes them with -DUSE_REFERENCE -I<reference tree>
REFERENCE_PROTOTYPES = ROOT / "tests" / "golden" / "abi_prototypes_reference.txt"


def _build(tmp, name, flags, link):
    exe = tmp / name
    cmd = ["gcc", "-std=gnu11", "-O0", "-w", str(ROOT / "tests" / "abi" / "abi_probe.c"), "-o", str(exe)] + flags
    if link:
        lib = ROOT / "aresdb_b200" / "lib"
        cmd += [f"-L{lib}", "-lalgorithm", "-lmem", f"-Wl,-rpath,{lib}"]
    else:
        cmd += ["-Wl,--unresolved-symbols=ignore-all"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_struct_layouts_and_enums_equal_the_reference_headers(tmp_path):
    ours = _build(tmp_path, "probe_ours", [f"-I{ROOT / 'include'}"], link=False)
    a = subprocess.run([str(ours)], capture_output=True, text=True).stdout
    assert a.count("\n") > 130
    assert a == REFERENCE_LAYOUT.read_text()


def prototype_digests(tmp, flags, header_dir: str) -> dict:
    """function name -> sha256 of the prototype gcc -aux-info prints for it (parameter types only, no names), for the
    functions declared in headers under header_dir."""
    aux = tmp / "aux.txt"
    r = subprocess.run(["gcc", "-std=gnu11", "-fsyntax-only", "-aux-info", str(aux), str(ROOT / "tests" / "abi" / "abi_probe.c")]
                       + flags, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    out = {}
    for line in aux.read_text().splitlines():
        m = re.match(r"/\* (\S+):\d+:\w+ \*/ (?:extern )?(.*);$", line.strip())
        if m and header_dir in m.group(1):
            out[re.search(r"(\w+) \(", m.group(2)).group(1)] = hashlib.sha256(m.group(2).encode()).hexdigest()
    return out


def test_function_prototypes_equal_the_reference_headers(tmp_path):
    ours = prototype_digests(tmp_path, [f"-I{ROOT / 'include'}"], "/include/aresdb_b200/")
    ref = dict(line.split() for line in REFERENCE_PROTOTYPES.read_text().splitlines())
    assert len(ref) > 30
    assert {n: ours.get(n) for n in ref} == ref


def test_project_header_build_links_against_the_b200_libraries(tmp_path):
    lib = ROOT / "aresdb_b200" / "lib" / "libalgorithm.so"
    if not lib.exists():
        pytest.skip("engine not built")
    exe = _build(tmp_path, "probe_link", [f"-I{ROOT / 'include'}"], link=True)
    r = subprocess.run([str(exe), "link"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "link symbols 10" in r.stdout and "link GetFlags" in r.stdout
