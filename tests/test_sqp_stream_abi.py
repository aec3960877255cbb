"""The ctypes mirror of sqpb200_sqp_stream (restartsqp_b200/sqp_device.py) against the header: field offsets and size as a C
compiler lays them out."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

from restartsqp_b200.sqp_device import SqpStream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("gcc") is None, reason="needs gcc")
def test_stream_descriptor_layout_matches_the_header(tmp_path):
    names = [f[0] for f in SqpStream._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sqpb200.h"\nint main(void) {\n' +
                   "".join('    printf("%s %%zu\\n", offsetof(sqpb200_sqp_stream, %s));\n' % (k, k) for k in names) +
                   '    printf("sizeof %zu\\n", sizeof(sqpb200_sqp_stream));\n    return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert {k: int(out[k]) for k in names} == {k: getattr(SqpStream, k).offset for k in names}
    assert int(out["sizeof"]) == C.sizeof(SqpStream)
