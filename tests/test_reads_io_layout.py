"""CPU: the ctypes mirror of struct elector_reads_io (elector_b200/poa.py) has the layout of include/elector_poa.h: a C file compiled
against the header prints sizeof and the offset of every field, and those equal the ctypes struct's."""
import ctypes
import os
import subprocess

from conftest import ROOT


def test_reads_io_mirror_matches_the_header(tmp_path):
    from elector_b200.poa import ReadsIoC
    names = [f[0] for f in ReadsIoC._fields_]
    src = tmp_path / "layout.c"
    src.write_text("#include <stddef.h>\n#include <stdio.h>\n#include \"elector_poa.h\"\nint main(void) {\n"
                   "  printf(\"sizeof %zu\\n\", sizeof(elector_reads_io));\n"
                   + "".join("  printf(\"%s %%zu\\n\", offsetof(elector_reads_io, %s));\n" % (n, n) for n in names)
                   + "  return 0;\n}\n")
    exe = str(tmp_path / "layout")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-o", exe, str(src)])
    got = dict(line.split() for line in subprocess.check_output([exe], text=True).splitlines())
    assert int(got.pop("sizeof")) == ctypes.sizeof(ReadsIoC)
    assert {n: int(v) for n, v in got.items()} == {n: getattr(ReadsIoC, n).offset for n in names}
