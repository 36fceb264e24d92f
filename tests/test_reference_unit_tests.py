"""The reference's own unit-test modules, unmodified, against the drop-in.

tests/golden/reference_tests/ holds byte-identical copies of
src/python/library/tests/test_cuda_shared_memory.py (DLPack in / out on GPU and CPU, numpy set ->
DLPack read, numpy set -> get_contents_as_numpy, BYTES through a CUDA region; needs torch + a GPU)
and test_shared_memory.py (SURVEY.md section 4).  Each is loaded with `client_b200` installed as
`tritonclient` and run by unittest in a fresh interpreter."""

import hashlib
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FIX = os.path.join(HERE, "golden", "reference_tests")
DIGESTS = os.path.join(HERE, "golden", "reference_digests.json")


def _run(module_file, timeout=300):
    runner = ("import sys, unittest, importlib.util; sys.path.insert(0, %r); import client_b200; client_b200.install_as_tritonclient(); "
              "spec = importlib.util.spec_from_file_location('ref_unit_tests', %r); "
              "mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod); "
              "res = unittest.TextTestRunner(verbosity=0).run(unittest.TestLoader().loadTestsFromModule(mod)); "
              "print('RAN', res.testsRun, len(res.failures), len(res.errors), len(res.skipped)); sys.exit(0 if res.wasSuccessful() else 1)"
              % (ROOT, os.path.join(FIX, module_file)))
    return subprocess.run([sys.executable, "-W", "ignore", "-c", runner], capture_output=True, text=True, timeout=timeout)


@pytest.mark.parametrize("name", ["test_cuda_shared_memory.py", "test_shared_memory.py"])
def test_fixture_copies_are_the_reference_files(name):
    """Each copy hashes to the digest taken from the reference's own file."""
    with open(DIGESTS) as fh:
        want = json.load(fh)["files"]["src/python/library/tests/" + name]
    with open(os.path.join(FIX, name), "rb") as fh:
        assert hashlib.sha256(fh.read()).hexdigest() == want


def test_reference_system_shared_memory_unit_tests_unmodified():
    r = _run("test_shared_memory.py")
    assert r.returncode == 0 and "RAN 7 0 0" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
def test_reference_cuda_shared_memory_unit_tests_unmodified():
    """test_cuda_shared_memory.py:42-164: DLPackTest (from_gpu, from_cpu) and NumpyTest
    (numpy -> DLPack, numpy -> numpy, BYTES) -- 5 tests, none skipped."""
    r = _run("test_cuda_shared_memory.py")
    assert r.returncode == 0 and "RAN 5 0 0 0" in r.stdout, r.stdout + r.stderr
