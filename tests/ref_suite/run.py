"""Runs the REFERENCE'S OWN test files against this package (needs the copy of the reference that build() stages
under oracle/_ref by oracle/make_ref.sh).

    python tests/ref_suite/run.py [test_file.py …] [pytest args…]

A scratch directory gets a generated package ``torchsnapshot`` whose ``__path__`` is
``[shims, <repo>/torchsnapshot_b200, <repo>/oracle/_ref/torchsnapshot]``: ``torchsnapshot.batcher``,
``.io_preparers.tensor``, ``.scheduler``, ``.snapshot`` … load OUR files (as a second, self-consistent copy of the
package under the reference's name), while helper modules we do not mirror (``test_utils``, ``uvm_tensor`` …) load the
reference's files, whose relative imports then bind to our modules.  Spawned worker processes (run_with_pet) import
the same generated package.  Nothing is copied from the reference: its test files are symlinked."""
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
OURS = os.path.join(REPO, "torchsnapshot_b200")
REF = os.path.join(REPO, "oracle", "_ref", "torchsnapshot")
REF_TESTS = os.path.join(REPO, "oracle", "_ref", "tests")
DEFAULT = [
    "test_flatten.py", "test_manifest.py", "test_chunked_tensor_io_preparer.py", "test_tensor_io_preparer.py", "test_batcher.py",
    "test_sharded_tensor_resharding.py", "test_sharded_tensor_io_preparer.py", "test_partitioner.py", "test_snapshot.py", "test_state_dict.py",
    "test_rng_state.py", "test_read_object.py", "test_replication_glob.py", "test_ddp.py", "test_async_take.py", "test_fs_storage_plugin.py",
    "test_serialization.py", "test_ddp_infer_replication.py", "test_ddp_replication_glob.py", "test_pg_wrapper.py",
]
# single-process files: fast enough for the regular CPU suite (tests/test_reference_suite.py)
FAST = [
    "test_flatten.py", "test_manifest.py", "test_serialization.py", "test_tensor_io_preparer.py", "test_batcher.py",
    "test_sharded_tensor_resharding.py", "test_state_dict.py", "test_rng_state.py", "test_fs_storage_plugin.py", "test_snapshot.py",
]

SHIMS = {
    # modules whose names exist in the reference but whose content lives elsewhere in this package
    "rng_state.py": "from .stateful import RNGState  # noqa: F401\n",
    "state_dict.py": "from .stateful import StateDict  # noqa: F401\n",
    "manifest_utils.py": (
        "from .manifest import (  # noqa: F401\n"
        "    is_container_entry, is_dict_entry, is_fully_replicated_entry, is_partially_replicated_entry,\n"
        "    is_replicated_entry, is_sharded_entry,\n)\n"
        "from .partitioner import replica_groups as _get_replicated_ranks  # noqa: F401\n"
    ),
}


def make_overlay(work: str) -> None:
    shims = os.path.join(work, "_shims")
    os.makedirs(shims)
    for name, body in SHIMS.items():
        with open(os.path.join(shims, name), "w") as f:
            f.write(body)
    pkg = os.path.join(work, "torchsnapshot")
    os.makedirs(pkg)
    with open(os.path.join(pkg, "__init__.py"), "w") as f:
        f.write(
            "import os\n"
            f"__path__ = [{shims!r}, {OURS!r}, {REF!r}]\n"
            f"_init = os.path.join({OURS!r}, '__init__.py')\n"
            "exec(compile(open(_init).read(), _init, 'exec'))\n"
        )


if __name__ == "__main__":
    if not os.path.isdir(REF_TESTS):
        print("oracle/_ref/tests not staged (oracle/make_ref.sh); nothing to run")
        sys.exit(0)
    import pytest

    work = tempfile.mkdtemp(prefix="ref_suite_")
    make_overlay(work)
    picked = [a for a in sys.argv[1:] if a.endswith(".py")] or (FAST if "--fast" in sys.argv else DEFAULT)
    extra = [a for a in sys.argv[1:] if not a.endswith(".py") and a != "--fast"]
    for f in picked:
        os.symlink(os.path.join(REF_TESTS, f), os.path.join(work, f))
    shutil.copy(os.path.join(HERE, "overlay_conftest.py"), os.path.join(work, "conftest.py"))
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
    sys.path.insert(0, work)
    os.environ["PYTHONPATH"] = work + os.pathsep + os.environ.get("PYTHONPATH", "")
    rc = pytest.main(["-q", "-p", "no:cacheprovider", "--rootdir", work, "-o", "addopts=", work] + extra)
    shutil.rmtree(work, ignore_errors=True)
    sys.exit(rc)
