"""Drop-in proof on the CPU: the original project's tests/test_pnode.py, restated in tests/_pnode_reference_tests.py, executed
as a script against this repo's `pnode` / `petsc4py` packages.  No GPU is needed: the device kernels are replaced by the
torch-CPU test double of tests/_fake_ops.py (the same comparisons run through the real kernels in
tests/test_gpu_generic.py::test_reference_rober_known_answers_on_gpu)."""
import importlib.util
import os
import sys

import pytest

REF_TEST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_pnode_reference_tests.py")


@pytest.fixture()
def ref_module(monkeypatch):
    from _fake_ops import patch_cpu
    from pnode_b200.options import Options

    patch_cpu(monkeypatch)
    monkeypatch.setattr(sys, "argv", ["test_pnode.py"])
    Options.clear_all()
    spec = importlib.util.spec_from_file_location("ref_test_pnode", REF_TEST)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)  # runs petsc4py.init(sys.argv + ...) with the file's own PETSc options
    assert mod.petsc_adjoint.__name__ == "pnode_b200.petsc_adjoint"
    return mod


@pytest.mark.parametrize("name", ["test_petsc_scalartype", "test_petsc_implicit_odesolver", "test_petsc_imex_odesolver",
                                  "test_petsc_explicit_odesolver"])
def test_reference_test_passes_against_the_drop_in(ref_module, name):
    from pnode_b200.options import Options

    # the file's own options reached the engine through petsc4py.init
    assert Options().getString("ts_adapt_type") == "none"
    assert Options().getString("ts_trajectory_type") == "memory"
    getattr(ref_module, name)()
