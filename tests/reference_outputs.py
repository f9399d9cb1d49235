"""What the reference's own sources computed on the inputs the tests build, kept as SHA-256 digests in
tests/golden/reference_outputs.json, so that every comparison with the reference runs on any checkout.

Where the reference libraries exist (oracle/_ref/, which oracle/Makefile builds from the reference tree), each comparison
also runs live against them.  `REFSRC_RECORD=1 python -m pytest tests/...` rewrites the record from those libraries."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.json")
RECORD = os.environ.get("REFSRC_RECORD") == "1"
_store = None
_recorded = set()      # keys written by this process: a key must not stand for two different outputs


def _load():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(PATH):
            with open(PATH) as f:
                _store = json.load(f)
    return _store


def _feed(h, x):
    if x is None:
        h.update(b"N")
    elif hasattr(x, "__dict__"):        # the views of _abi / oracle.ref: their arrays and scalars
        _feed(h, vars(x))
    elif isinstance(x, dict):
        h.update(b"{%d" % len(x))
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    elif isinstance(x, (tuple, list)):
        h.update(b"(%d" % len(x))
        for v in x:
            _feed(h, v)
    else:
        a = np.ascontiguousarray(x)
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())


def digest(x) -> str:
    """SHA-256 over dtypes, shapes and bytes of arrays, scalars, None and nested tuples / lists / dicts / objects of
    them."""
    h = hashlib.sha256()
    _feed(h, x)
    return h.hexdigest()


class Reference:
    """The reference's outputs for one test: `live` says whether its library is loadable here."""

    def __init__(self, test: str, live: bool):
        self.test, self.live = test, live
        if RECORD and not live:
            raise RuntimeError("REFSRC_RECORD=1 needs the reference libraries under oracle/_ref")

    def _key(self, tag):
        return "%s/%s" % (self.test, tag)

    def same(self, tag, mine, ref=None):
        """`mine` must be bit for bit what the reference computed for `tag`: live through `ref()` (a callable running the
        reference) where its library exists, and always against the recorded digest."""
        key, d = self._key(tag), digest(mine)
        if self.live and ref is not None:
            assert digest(ref()) == d, (key, "differs from the reference's own sources")
        store = _load()
        if RECORD:
            assert key not in _recorded or store[key] == d, (key, "recorded twice with different outputs")
            _recorded.add(key)
            store[key] = d
            self._save()
        else:
            assert key in store, (key, "no recorded reference output")
            assert store[key] == d, (key, "differs from the recorded output of the reference's own sources")

    def value(self, tag, ref):
        """A reference output the test feeds on (a nested list of numbers): live from `ref()` where the library exists,
        otherwise the recorded one; live and recorded must agree."""
        key = self._key(tag) + ":value"
        store = _load()
        if self.live:
            v = json.loads(json.dumps(ref()))
            if RECORD:
                store[key] = v
                self._save()
            else:
                assert store.get(key) == v, (key, "differs from the recorded output of the reference's own sources")
            return v
        assert key in store, (key, "no recorded reference output")
        return store[key]

    @staticmethod
    def _save():
        with open(PATH, "w") as f:
            json.dump(_store, f, indent=0, sort_keys=True)
            f.write("\n")
