"""The ctypes mirror of sasa_b200_pair_sums lays out like the C compiler lays out the header's struct (no device needed)."""
import ctypes as C
import os
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pair_sums_layout_matches_header():
    from rustsasa_b200 import _lib
    fields = [name for name, _ in _lib.PairSums._fields_]
    assert fields == ["n_labels", "pair_area", "seg_pair_area"]
    prog = ('#include <stddef.h>\n#include <stdio.h>\n#include "sasa_b200.h"\nint main(void){printf("%zu'
            + ' %zu' * len(fields) + '\\n", sizeof(sasa_b200_pair_sums)'
            + "".join(f", offsetof(sasa_b200_pair_sums, {f})" for f in fields) + ');return 0;}\n')
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "t.c"), os.path.join(d, "t")
        with open(src, "w") as fh:
            fh.write(prog)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", exe, src], check=True)
        out = [int(x) for x in subprocess.run([exe], check=True, stdout=subprocess.PIPE, text=True).stdout.split()]
    assert out == [C.sizeof(_lib.PairSums)] + [getattr(_lib.PairSums, f).offset for f in fields]
