"""Runs the compiled SparsifiedGP drop-in test (tests/cpp/sparse_dropin_test.cpp): the reference's own
limbo::model::SparsifiedGP and limbo::model::MultiGP<Params, SparsifiedGP, ...> next to limbo_b200::model::SparsifiedGP and
MultiGP over it.  The binary is built where the reference's sources exist (__graft_entry__.build()) and lies in
oracle/_ref/."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "oracle", "_ref", "sparse_dropin_test")


@pytest.mark.gpu
def test_reference_sparsified_gp_next_to_b200():
    if not os.path.exists(BIN):
        pytest.skip("oracle/_ref/sparse_dropin_test not built (needs the reference's sources at build time)")
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "limbo_b200", "lib") + ":" + os.environ.get("LD_LIBRARY_PATH", ""))
    r = subprocess.run([BIN], capture_output=True, text=True, timeout=600, env=env)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "SPARSE DROPIN OK" in r.stdout, r.stdout + r.stderr
