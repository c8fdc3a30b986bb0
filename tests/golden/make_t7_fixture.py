"""Builds the fixture that pins bot7_b200/t7.py against the reference's own Torch7 data file.

examples/data/iris_test30.t7 (reference repository, 6528 bytes: a Lua table of four DoubleTensors written by
torch.save) is the only binary-format artefact the reference ships.  The file itself is not copied: the fixture
holds what this repository's reader extracts from it (the four arrays, in file order) plus the SHA-256 and the
length of the original bytes.  tests/test_t7.py re-serialises the arrays with this repository's writer and
requires the digest of the result to equal the digest of the reference file, i.e. the writer is byte-exact and the
reader (which produced the arrays, and which reads the re-serialised bytes back) is consistent with it.
Run (with a checkout of the reference): BOT7_REFERENCE=<bot7 checkout> python tests/golden/make_t7_fixture.py
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from bot7_b200 import t7  # noqa: E402

if __name__ == "__main__":
    ref = os.environ.get("BOT7_REFERENCE", "")
    if not os.path.isdir(ref):
        sys.exit("set BOT7_REFERENCE to a checkout of the reference bot7 source")
    raw = open(os.path.join(ref, "examples", "data", "iris_test30.t7"), "rb").read()
    table = t7.loads(raw)
    assert t7.dumps({k: np.array(v) for k, v in table.items()}) == raw
    out = os.path.join(HERE, "ref_iris_test30.npz")
    np.savez_compressed(out, order=np.array(list(table)), sha256=np.array(hashlib.sha256(raw).hexdigest()), nbytes=np.array(len(raw)),
                        **{k: np.array(v) for k, v in table.items()})
    print(out, hashlib.sha256(raw).hexdigest(), len(raw))
