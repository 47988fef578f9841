"""Stored outputs of the reference project's own builds, for the tests that compare with them.

oracle/build_ref.py and oracle/build_ref_cuda.py compile the reference's CPU and CUDA extensions into oracle/_ref/ only
where the reference's sources are at hand.  Everywhere else a test compares with what those builds returned for the same
inputs, stored under tests/golden/: the whole array where the test needs it as an input, otherwise the SHA-256 of its
bytes with its shape, dtype and first values (bit-exact, like torch.equal, and a failure shows what differs).  Where the
builds are present, the tests compare with them directly and check that they still return the stored outputs (where
those are deterministic: the reference's CPU sampler draws unseeded).  QV_RECORD_REF_GOLDEN=1 makes them rewrite the
stored file from the builds instead.
"""
import hashlib
import json
import os

import numpy as np

RECORD = os.environ.get("QV_RECORD_REF_GOLDEN") == "1"


def _host(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a)


def digest(a):
    a = _host(a)
    return {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": hashlib.sha256(a.tobytes()).hexdigest(),
            "head": a.reshape(-1)[:8].tolist()}


class ReferenceOutputs:
    """The reference's outputs for one test module: `live` is the loaded reference build, or None."""

    def __init__(self, path, live, source, deterministic=True):
        self.path, self.live, self.source, self.deterministic = path, live, source, deterministic
        self.record = RECORD and live is not None
        self.entries = {} if self.record else json.load(open(path))["entries"]

    def check(self, key, ours, theirs=None):
        """ours: {name: array} computed by this project; theirs: the same names from the live build (None without it)."""
        for name, a in ours.items():
            k = f"{key}/{name}"
            if theirs is not None:
                want = digest(theirs[name])
                if self.record:
                    self.entries[k] = want
                elif self.deterministic:
                    assert want == self.entries[k], f"{k}: the reference build no longer returns the stored output"
            else:
                want = self.entries[k]
            got = digest(a)
            assert got == want, f"{k}: got {got}, the reference returned {want}"

    def arrays(self, key, theirs=None):
        """The reference's arrays {name: int64 array}: from the live build (recorded whole when recording), else stored."""
        if theirs is not None:
            theirs = {name: _host(a) for name, a in theirs.items()}
            if self.record:
                self.entries[key] = {name: a.tolist() for name, a in theirs.items()}
            return theirs
        return {name: np.array(v, dtype=np.int64) for name, v in self.entries[key].items()}

    def save(self):
        if self.record:
            with open(self.path, "w") as f:
                json.dump({"source": self.source, "entries": self.entries}, f, separators=(",", ":"))
