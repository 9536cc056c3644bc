"""CPU check that the ctypes mirror of team_loss_shard (team_b200/capi.py) has the size and field offsets of the C struct
in include/team_b200.h (a small C program compiled with gcc prints them, as in test_abi_layout.py)."""
import ctypes
import os
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_loss_shard_mirror_matches_the_c_header():
    from team_b200 import capi
    fields = [n for n, _ in capi.LossShard._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "team_b200.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(team_loss_shard));']
    lines += [f'  printf("{f} %zu\\n", offsetof(team_loss_shard, {f}));' for f in fields]
    lines += ["  return 0;", "}"]
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "abi.c"), os.path.join(td, "abi")
        with open(src, "w") as fh:
            fh.write("\n".join(lines))
        subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    got = {k: int(v) for k, v in (ln.split() for ln in out.splitlines())}
    assert ctypes.sizeof(capi.LossShard) == got["size"], (ctypes.sizeof(capi.LossShard), got["size"])
    for f in fields:
        assert getattr(capi.LossShard, f).offset == got[f], (f, getattr(capi.LossShard, f).offset, got[f])
