"""CPU tests: the library has no hidden configurations. The CUDA sources read no environment variables, and the
Python package reads exactly the ones listed here, so every code path that runs is one the suite builds, tests and
times. A new switch has to be added to this list on purpose."""
import ast
import glob
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PY_ENV_VARS = {
    "SPNET_B200_POISON",    # fill fresh activation buffers with NaN: a read of memory nothing wrote fails loudly
    "SPNET_B200_NO_GRAPH",  # predict / fit run eagerly instead of replaying a captured CUDA graph
    "SPNET_B200_DP_COMM",   # precision of the data-parallel gradient all-reduce (bf16 / fp32)
    "SPNET_B200_DP_TRACE",  # per-stream event timeline of data-parallel steps (reported by bench.py)
}


def test_cuda_sources_read_no_environment_variables():
    srcs = sorted(glob.glob(os.path.join(ROOT, "spnet_b200", "csrc", "*.cu"))
                  + glob.glob(os.path.join(ROOT, "spnet_b200", "csrc", "*.cuh")))
    assert srcs
    assert [os.path.basename(p) for p in srcs if "getenv" in open(p).read()] == []


def _is_environ(node):
    return isinstance(node, ast.Attribute) and node.attr == "environ"


def _key(node):
    return node.value if isinstance(node, ast.Constant) and isinstance(node.value, str) else "<not a literal>"


def env_vars_read(path):
    """Names read by os.environ.get(...) (or any other os.environ method), os.getenv(...), os.environ[...] and
    `... in os.environ`."""
    names = set()
    for node in ast.walk(ast.parse(open(path).read(), path)):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and (
                node.func.attr == "getenv" or _is_environ(node.func.value)):
            names.add(_key(node.args[0]) if node.args else "<not a literal>")
        elif isinstance(node, ast.Subscript) and _is_environ(node.value):
            names.add(_key(node.slice))
        elif isinstance(node, ast.Compare) and any(_is_environ(c) for c in node.comparators):
            names.add(_key(node.left))
    return names


def test_python_package_reads_only_the_listed_environment_variables():
    files = sorted(glob.glob(os.path.join(ROOT, "spnet_b200", "*.py")))
    assert files
    seen = {}
    for p in files:
        for name in env_vars_read(p):
            seen.setdefault(name, []).append(os.path.basename(p))
    assert set(seen) == PY_ENV_VARS, seen
