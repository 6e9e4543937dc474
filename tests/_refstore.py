"""What the reference's own code answered for the inputs of the differential tests, stored under tests/golden/ so that
these tests hold on any machine, with or without the reference libraries of oracle/_ref.

    want(store, key, live)   the value recorded for `key` in tests/golden/ref_<store>.json.  With REF_RECORD=<dir> in the
                             environment it calls `live()` -- the reference itself, through oracle/_ref -- instead, and
                             writes the answer to <dir>/ref_<store>.json (copy that file to tests/golden/ to keep it).

A value is anything JSON holds; arrays go in as digest(array), so a large output costs 71 bytes and is still compared
exactly.  Regenerate with e.g. `REF_RECORD=/tmp/ref python -m pytest tests/test_oracle_vs_ref.py` (the GPU stores on a
GPU machine with `-m gpu`)."""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_stores = {}


def digest(a):
    """SHA-256 of an array's element type and bytes"""
    a = np.ascontiguousarray(a)
    return "sha256:" + hashlib.sha256(a.dtype.str.encode() + a.tobytes()).hexdigest()


def want(store, key, live):
    record = os.environ.get("REF_RECORD")
    if record:
        value = json.loads(json.dumps(live()))     # as it will read back (tuples become lists)
        path = os.path.join(record, "ref_%s.json" % store)
        os.makedirs(record, exist_ok=True)
        data = json.load(open(path)) if os.path.exists(path) else {}
        data[key] = value
        with open(path, "w") as f:   # one answer per line
            f.write("{\n%s\n}\n" % ",\n".join("%s: %s" % (json.dumps(k), json.dumps(data[k])) for k in sorted(data)))
        return value
    if store not in _stores:
        with open(os.path.join(GOLDEN, "ref_%s.json" % store)) as f:
            _stores[store] = json.load(f)
    assert key in _stores[store], "no recorded reference answer for %s in tests/golden/ref_%s.json" % (key, store)
    return _stores[store][key]
