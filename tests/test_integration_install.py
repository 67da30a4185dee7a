"""(The reference's own async_take cannot run in this container: T:dist_store.py:69 unpacks a 4-tuple from an
IPv4 getsockname(); SURVEY.md §4.  async_take is covered through this package's Snapshot instead.)

`torchsnapshot_b200.install()` puts the engine underneath the UNMODIFIED reference: its own
Snapshot.take/restore keep producing the golden bytes, but the raw tensor traffic goes through
libtsnap_b200.so.  Needs the copy of the reference that build() stages under oracle/_ref (oracle/make_ref.sh)."""
import os
import sys

import pytest
import torch

from tests.cases import CASES, apply_knobs
from tests.test_parity_cpu import _golden, assert_matches_golden
from tests.util import snapshot_digest, wire_bytes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# staged by build() (oracle/make_ref.sh); the staged copy travels with the working tree
REF_PARENT = os.path.join(ROOT, "oracle", "_ref")
pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(REF_PARENT, "torchsnapshot")), reason="reference not staged (oracle/make_ref.sh)")


def test_staged_reference_is_the_unmodified_tree():
    """oracle/_ref must be a verbatim copy: every file's sha256 equals the one oracle/make_ref.sh recorded from the
    source tree at staging time, and no file was added."""
    import hashlib

    staged = os.path.join(REF_PARENT, "torchsnapshot")
    want = dict(reversed(ln.split(None, 1)) for ln in open(os.path.join(REF_PARENT, "MANIFEST.sha256")).read().splitlines() if ln.strip())
    want = {rel.strip(): digest for rel, digest in want.items()}
    assert len(want) > 40
    for rel, digest in want.items():
        assert hashlib.sha256(open(os.path.join(staged, rel), "rb").read()).hexdigest() == digest, rel
    have = {"./" + os.path.relpath(os.path.join(dp, f), staged) for dp, _, fs in os.walk(staged) if "__pycache__" not in dp for f in fs}
    assert have == set(want)


@pytest.fixture()
def ref():
    sys.path.insert(0, REF_PARENT)
    os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
    try:
        import torchsnapshot
    finally:
        sys.path.remove(REF_PARENT)
    import torchsnapshot_b200 as B

    B.install(torchsnapshot)
    yield torchsnapshot
    B.uninstall()


@pytest.mark.parametrize("name", ["dtypes_and_views", "chunked_slabbed", "slabs", "model_adam"])
def test_reference_api_runs_on_the_engine(ref, name, tmp_path):
    import torchsnapshot_b200 as B
    from torchsnapshot_b200.flatten import flatten

    build, knobs = CASES[name]
    state = build("cpu")
    eng = B.get_engine(-1)
    before = eng.stats()["bytes_written"]
    with apply_knobs(knobs):
        snap = ref.Snapshot.take(str(tmp_path / "snap"), {"state": ref.StateDict(**state)})
        assert eng.stats()["bytes_written"] > before, "the engine was not on the path"
        assert_matches_golden(snapshot_digest(str(tmp_path / "snap")), _golden(name))
        target = build("cpu")
        for v in flatten(target, "x")[1].values():
            if isinstance(v, torch.Tensor):
                v.zero_()
        before_r = eng.stats()["bytes_read"]
        tgt = ref.StateDict(**target)
        snap.restore({"state": tgt})
        assert eng.stats()["bytes_read"] > before_r
    a, b = flatten(state, "x")[1], flatten(dict(tgt), "x")[1]
    for k in a:
        if isinstance(a[k], torch.Tensor):
            assert wire_bytes(a[k]) == wire_bytes(b[k]), k
        else:
            assert a[k] == b[k], k


def test_storage_plugins_entry_point(ref, tmp_path, monkeypatch):
    """pyproject.toml registers b200fs in the reference's `storage_plugins` entry-point group
    (T:storage_plugin.py:56-67); resolve it the way the reference does and take/restore through it."""
    import importlib
    import tomllib

    import torchsnapshot_b200 as B

    B.uninstall()
    proj = tomllib.load(open(os.path.join(ROOT, "pyproject.toml"), "rb"))
    target = proj["project"]["entry-points"]["storage_plugins"]["b200fs"]
    mod, attr = target.split(":")
    factory = getattr(importlib.import_module(mod), attr)

    class EP:  # what importlib.metadata hands the reference after `pip install`
        name, value = "b200fs", target

        @staticmethod
        def load():
            return factory

    sp = importlib.import_module(ref.__name__ + ".storage_plugin")
    monkeypatch.setattr(sp, "entry_points", lambda group=None: [EP] if group == "storage_plugins" else [])
    build, knobs = CASES["slabs"]
    state = build("cpu")
    eng = B.get_engine(-1)
    w0 = eng.stats()["bytes_written"]
    with apply_knobs(knobs):
        snap = ref.Snapshot.take("b200fs://" + str(tmp_path / "snap"), {"state": ref.StateDict(**state)})
        assert eng.stats()["bytes_written"] > w0, "the engine was not put underneath the reference"
        assert_matches_golden(snapshot_digest(str(tmp_path / "snap")), _golden("slabs"))
        tgt = ref.StateDict(**{k: torch.zeros_like(v) if isinstance(v, torch.Tensor) else v for k, v in state.items()})
        snap.restore({"state": tgt})
    for k, v in state.items():
        if isinstance(v, torch.Tensor):
            assert wire_bytes(v) == wire_bytes(tgt[k]), k
