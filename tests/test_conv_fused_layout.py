"""The ctypes mirrors of UbConvSeg / UbConvEpilogue / UbConvPlanInfo (unet.cu_b200/__init__.py) have the layout of
include/unet_b200.h: sizeof and every field's offset, printed by a tiny probe compiled against the header.  CPU suite,
needs nvcc (no GPU, the library is not loaded)."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = shutil.which("nvcc")


@pytest.mark.skipif(not NVCC, reason="needs nvcc")
def test_conv_fused_structs_match_the_header(tmp_path):
    import __graft_entry__ as ge
    ub = ge.load_package()
    structs = [ub.UbConvSeg, ub.UbConvEpilogue, ub.UbConvPlanInfo]
    lines = []
    for s in structs:
        lines.append(f'std::printf("{s.__name__} %zu\\n", sizeof({s.__name__}));')
        for f, _ in s._fields_:
            lines.append(f'std::printf("{s.__name__}.{f} %zu\\n", offsetof({s.__name__}, {f}));')
    src = tmp_path / "probe.cpp"
    src.write_text('#include <cstddef>\n#include <cstdio>\n#include "unet_b200.h"\nint main() {\n' + "\n".join(lines) +
                   "\nreturn 0;\n}\n")
    r = subprocess.run([NVCC, "-std=c++17", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(tmp_path / "probe")],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    got = subprocess.run([str(tmp_path / "probe")], stdout=subprocess.PIPE, text=True, check=True).stdout.split("\n")
    want = []
    for s in structs:
        want.append(f"{s.__name__} {C.sizeof(s)}")
        want += [f"{s.__name__}.{f} {getattr(s, f).offset}" for f, _ in s._fields_]
    assert got[:-1] == want
