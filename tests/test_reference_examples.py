"""The reference's own example scripts, UNMODIFIED, run against the drop-in package
(`client_b200.install_as_tritonclient()`) and the mock server: every script ends with its own
value checks and exits non-zero on a mismatch (SURVEY.md section 4, "examples as tests").
The Python example scripts are read from the reference's source tree; where it is absent those
tests skip.  The C++ programs run from the binaries build() compiled under oracle/_ref/cc_examples/.
Not run: the CUDA shared memory examples (GPU tests restate them), the model-control examples
(server repository semantics), simple_http_infer_client.py (imports gevent itself, absent here),
ensemble_image_client.py / image_client.py over HTTP (import attrdict, absent here)."""

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from test_loopback import start_server

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXAMPLES = "/root/reference/src/python/examples"
RUNNER = ("import sys; sys.path.insert(0, %r); import client_b200; client_b200.install_as_tritonclient(); "
          "import runpy; sys.argv = sys.argv[1:]; runpy.run_path(sys.argv[0], run_name='__main__')" % ROOT)

SCRIPTS = [
    "grpc_client.py", "grpc_explicit_byte_content_client.py", "grpc_explicit_int8_content_client.py",
    "grpc_explicit_int_content_client.py", "reuse_infer_objects_client.py", "simple_grpc_aio_infer_client.py",
    "simple_grpc_aio_sequence_stream_infer_client.py", "simple_grpc_async_infer_client.py",
    "simple_grpc_custom_args_client.py", "simple_grpc_custom_repeat.py", "simple_grpc_health_metadata.py",
    "simple_grpc_infer_client.py", "simple_grpc_keepalive_client.py", "simple_grpc_sequence_stream_infer_client.py",
    "simple_grpc_sequence_sync_infer_client.py", "simple_grpc_shm_client.py", "simple_grpc_shm_string_client.py",
    "simple_grpc_string_infer_client.py", "simple_http_aio_infer_client.py", "simple_http_async_infer_client.py",
    "simple_http_health_metadata.py", "simple_http_sequence_sync_infer_client.py", "simple_http_shm_client.py",
    "simple_http_shm_string_client.py", "simple_http_string_infer_client.py",
]
IMAGE_RUNS = [
    ("image_client.py", ["-m", "densenet_onnx", "-s", "INCEPTION", "-c", "3", "-i", "grpc"]),
    ("image_client.py", ["-m", "densenet_onnx", "-s", "VGG", "-c", "2", "-i", "grpc", "--streaming"]),
    ("image_client.py", ["-m", "densenet_onnx", "-s", "NONE", "-c", "1", "-i", "grpc", "-a"]),
    ("grpc_image_client.py", ["-m", "densenet_onnx", "-s", "INCEPTION", "-c", "3"]),
]

# the scripts are the reference's own sources, which the repository does not carry
needs_reference = pytest.mark.skipif(not os.path.isdir(EXAMPLES), reason="the reference's Python examples are absent")


@pytest.fixture(scope="module")
def outcomes(tmp_path_factory):
    from PIL import Image

    img = str(tmp_path_factory.mktemp("img") / "photo.png")
    Image.fromarray(np.random.default_rng(0).integers(0, 256, (300, 400, 3), dtype=np.uint8)).save(img)
    proc, http_port, grpc_port = start_server()
    jobs = []
    for name in SCRIPTS:
        port = grpc_port if name.startswith(("grpc_", "simple_grpc")) else http_port
        jobs.append((name, [os.path.join(EXAMPLES, name), "-u", "127.0.0.1:%d" % port]))
    for name, args in IMAGE_RUNS:
        jobs.append(("%s %s" % (name, " ".join(args)), [os.path.join(EXAMPLES, name)] + args + ["-u", "127.0.0.1:%d" % grpc_port, img]))

    def run(job):
        label, argv = job
        try:
            r = subprocess.run([sys.executable, "-c", RUNNER] + argv, capture_output=True, text=True, timeout=120, cwd=str(tmp_path_factory.getbasetemp()))
            return label, r.returncode, (r.stdout + r.stderr)[-1500:]
        except subprocess.TimeoutExpired:
            return label, -1, "timeout"

    # the shared memory examples all use the same POSIX keys and region names: one after another
    uses_shm = lambda label: "shm" in label or label.startswith("reuse_infer_objects")  # noqa: E731
    serial = [j for j in jobs if uses_shm(j[0])]
    parallel = [j for j in jobs if not uses_shm(j[0])]
    try:
        with ThreadPoolExecutor(max_workers=6) as pool:
            chain = pool.submit(lambda: [run(j) for j in serial])
            results = {label: (rc, tail) for label, rc, tail in pool.map(run, parallel)}
            results.update({label: (rc, tail) for label, rc, tail in chain.result()})
    finally:
        proc.terminate()
        proc.wait(10)
    return results


@needs_reference
@pytest.mark.parametrize("label", SCRIPTS + ["%s %s" % (n, " ".join(a)) for n, a in IMAGE_RUNS])
def test_unmodified_reference_example(outcomes, label):
    rc, tail = outcomes[label]
    assert rc == 0, tail
    assert "FAILED" not in tail, tail


# ---- the same gRPC examples with infer() on the native transport (TB200_GRPC_TRANSPORT=native) --
NATIVE_TRANSPORT_SCRIPTS = [
    "grpc_client.py", "grpc_explicit_byte_content_client.py", "grpc_explicit_int8_content_client.py", "grpc_explicit_int_content_client.py",
    "simple_grpc_infer_client.py", "simple_grpc_string_infer_client.py", "simple_grpc_sequence_sync_infer_client.py",
    "simple_grpc_health_metadata.py", "simple_grpc_keepalive_client.py", "simple_grpc_custom_args_client.py",
]


@pytest.fixture(scope="module")
def native_transport_outcomes(tmp_path_factory):
    proc, _, grpc_port = start_server()
    env = dict(os.environ, TB200_GRPC_TRANSPORT="native")

    def run(name):
        try:
            r = subprocess.run([sys.executable, "-c", RUNNER, os.path.join(EXAMPLES, name), "-u", "127.0.0.1:%d" % grpc_port],
                               capture_output=True, text=True, timeout=120, cwd=str(tmp_path_factory.getbasetemp()), env=env)
            return name, (r.returncode, (r.stdout + r.stderr)[-1500:])
        except subprocess.TimeoutExpired:
            return name, (-1, "timeout")

    try:
        with ThreadPoolExecutor(max_workers=5) as pool:
            return dict(pool.map(run, NATIVE_TRANSPORT_SCRIPTS))
    finally:
        proc.terminate()
        proc.wait(10)


@needs_reference
@pytest.mark.parametrize("name", NATIVE_TRANSPORT_SCRIPTS)
def test_unmodified_reference_example_on_the_native_grpc_transport(native_transport_outcomes, name):
    """The examples whose inferences are synchronous infer() calls, run with the drop-in's native
    HTTP/2 transport selected through the environment: same PASS / exit 0."""
    rc, tail = native_transport_outcomes[name]
    assert rc == 0, tail
    assert "FAILED" not in tail, tail


# ---- the reference's C++ examples, compiled unmodified against client_b200/cpp ----------------
CC_OUT = os.path.join(ROOT, "oracle", "_ref", "cc_examples")
CC_EXAMPLES = {
    "simple_http_infer_client": "PASS : Infer",
    "simple_http_async_infer_client": "PASS : Async Infer",
    "simple_http_string_infer_client": "PASS : String Infer",
    "simple_http_shm_client": "PASS : System Shared Memory",
    "simple_http_sequence_sync_infer_client": "[7] 1 : -1 : -1",
    # gRPC front end (client_b200/cpp/tb200_grpc_client.h: own HTTP/2 framing + message classes)
    "simple_grpc_infer_client": "PASS : Infer",
    "simple_grpc_async_infer_client": "PASS : Async Infer",
    "simple_grpc_string_infer_client": "PASS : String Infer",
    "simple_grpc_shm_client": "PASS : System Shared Memory",
    "simple_grpc_health_metadata": "Request for unknown model: 'wrong_model_name' is not found",
    "simple_grpc_sequence_sync_infer_client": "[7] 1 : -1 : -1",
    "simple_grpc_sequence_stream_infer_client": "[7] 1 : -1 : -1",
    "simple_grpc_keepalive_client": "PASS : KeepAlive",
    "simple_grpc_custom_args_client": "PASS : CustomArgs",
    "simple_grpc_custom_repeat": "",
    # both front ends in one program (-i http | grpc), system shared memory, objects reused across calls
    "reuse_infer_objects_client": "15 - 1 = 14",
    "reuse_infer_objects_client:grpc": "15 - 1 = 14",
}


@pytest.fixture(scope="module")
def cc_binaries():
    """{name: path}: built from the reference's sources where they are present, otherwise the
    binaries an earlier build() left under oracle/_ref/cc_examples/ (they travel with the tree)."""
    from oracle.build_ref_examples import build_ref_examples

    built = build_ref_examples()
    if not built and os.path.isdir(CC_OUT):
        built = {f: os.path.join(CC_OUT, f) for f in os.listdir(CC_OUT) if os.access(os.path.join(CC_OUT, f), os.X_OK)}
    return built


def _cc_binary(cc_binaries, name):
    if name not in cc_binaries:
        pytest.skip("oracle/_ref/cc_examples/%s was not built: no reference source tree at build time" % name)
    return cc_binaries[name]


@pytest.fixture(scope="module")
def cc_server():
    proc, http_port, grpc_port = start_server()
    yield {"http": "127.0.0.1:%d" % http_port, "grpc": "127.0.0.1:%d" % grpc_port}
    proc.terminate()
    proc.wait(10)


@pytest.mark.parametrize("name", sorted(CC_EXAMPLES))
def test_unmodified_reference_cc_example(cc_binaries, cc_server, name):
    """src/c++/examples/<name>.cc compiled as is against compat/{http,grpc}_client.h +
    libtb200client.so (oracle/build_ref_examples.py) and run against the mock server's models;
    the programs end with their own value checks."""
    exe, _, variant = name.partition(":")
    path = _cc_binary(cc_binaries, exe)
    grpc = "_grpc_" in exe or variant == "grpc"
    url = cc_server["grpc" if grpc else "http"]
    r = subprocess.run([path, "-u", url] + (["-i", "grpc"] if variant == "grpc" else []), capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and CC_EXAMPLES[name] in r.stdout + r.stderr, r.stdout[-800:] + r.stderr[-400:]


def test_reference_client_timeout_test_unmodified(cc_binaries):
    """src/c++/tests/client_timeout_test.cc (the reference's own timeout test program, compiled as
    is): sync / async / streaming over gRPC and sync / async over HTTP succeed with a generous
    client time-out and fail with the reference's "Deadline Exceeded" when the model takes 300 ms
    and the client allows 50 ms."""
    exe = _cc_binary(cc_binaries, "client_timeout_test")
    modes = (["-i", "grpc"], ["-i", "grpc", "-a"], ["-i", "grpc", "-s"], ["-i", "http"], ["-i", "http", "-a"])
    for extra, timeout_us, rc in (((), "5000000", 0), (("--delay-us", "300000"), "50000", 1)):
        proc, http_port, grpc_port = start_server(extra)
        try:
            for mode in modes:
                url = "127.0.0.1:%d" % (grpc_port if "grpc" in mode else http_port)
                r = subprocess.run([exe, "-u", url, "-t", timeout_us] + mode, capture_output=True, text=True, timeout=60)
                assert r.returncode == rc, (mode, r.stdout[-300:], r.stderr[-300:])
                if rc and "-s" not in mode:
                    assert "Deadline Exceeded" in r.stderr, (mode, r.stderr[-300:])
        finally:
            proc.terminate()
            proc.wait(10)


def test_reference_memory_leak_test_unmodified(cc_binaries, cc_server):
    """src/c++/tests/memory_leak_test.cc (compiled as is; the reference runs it under valgrind):
    200 vs 2000 repetitions, new client per repetition and one reused client, over HTTP and gRPC --
    the peak resident set must not grow with the repetition count."""
    exe = _cc_binary(cc_binaries, "memory_leak_test")

    def peak_kb(args):
        code = ("import resource, subprocess, sys; r = subprocess.run(%r, capture_output=True); "
                "print(r.returncode, resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss)" % (args,))
        rc, kb = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300).stdout.split()
        assert rc == "0", args
        return int(kb)

    for proto in ("http", "grpc"):
        for flag in ([], ["-R"]):
            base = [exe, "-u", cc_server[proto], "-i", proto]
            few, many = peak_kb(base + ["-r", "200"] + flag), peak_kb(base + ["-r", "2000"] + flag)
            assert many - few < 2048, (proto, flag, few, many)


def test_reference_unit_tests_for_system_shared_memory_unmodified():
    """src/python/library/tests/test_shared_memory.py (the reference's own unittest module, carried
    byte for byte as tests/golden/reference_tests/test_shared_memory.py) loaded as is with the
    drop-in aliased as `tritonclient`: the same run as
    test_reference_unit_tests.py::test_reference_system_shared_memory_unit_tests_unmodified."""
    from test_reference_unit_tests import _run

    r = _run("test_shared_memory.py", timeout=120)
    assert r.returncode == 0 and "RAN 7 0 0" in r.stdout, r.stdout + r.stderr
