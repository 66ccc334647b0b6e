"""The head of an environment record (aom_env_head of include/aomarl.h) has the layout lib.ENV_HEAD reads."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROGRAM = r"""
#include <stddef.h>
#include <stdio.h>
#include "aomarl.h"
#define F(name) printf("%s %zu\n", #name, offsetof(aom_env_head, name));
int main(void) {
  printf("size %zu\n", sizeof(aom_env_head));
  F(magic) F(bytes) F(fingerprint) F(frame) F(step) F(le_n) F(first) F(n_layers) F(acc) F(wind) F(amp) F(noise)
  F(nphotons) F(gain) F(reserved)
  return 0;
}
"""


def test_env_head_layout(tmp_path):
    from ao_marl_b200.lib import ENV_HEAD
    src, exe = tmp_path / "head.c", tmp_path / "head"
    src.write_text(PROGRAM)
    try:
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    except FileNotFoundError:
        pytest.skip("no C compiler")
    out = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(out.pop("size")) == ENV_HEAD.itemsize
    for name, off in out.items():
        assert ENV_HEAD.fields[name][1] == int(off), name
