import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: takes more than a few seconds on CPU")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O
    O.build()
    return O


class Recorded:
    """Digests of outputs that the tests compare with the reference sources in tape mode (oracle/_ref), stored in
    tests/golden/recorded_outputs.json so that those comparisons also run where the reference is not built.  A
    digest holds a case's configuration, its counters and sha256 of every array or file it compares.

    The entries are digests of this project's outputs (restatement, engine, host program) on those cases, not of
    the reference's.  RACH_RECORD_OUTPUTS=<file> rewrites them: that mode refuses to start unless every reference
    build is present, so each test's live comparison with the reference runs in the same session, and it writes
    <file> only if every test of the session passed.  The entries committed now were recorded without the reference
    builds (its sources are not part of this repository), from the code of a commit whose suite had compared the
    same cases with those builds and found them equal; a run with the reference builds confirms them."""
    PATH = os.path.join(ROOT, "tests", "golden", "recorded_outputs.json")
    REF_LIBS = ("libref_w.so", "libref_b.so", "libref_n.so", "libref_n2.so", "libref_u0.so")

    def __init__(self):
        import json
        self.out = os.environ.get("RACH_RECORD_OUTPUTS")
        if self.out:
            missing = [f for f in self.REF_LIBS if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", f))]
            if missing:
                raise pytest.UsageError("RACH_RECORD_OUTPUTS records only next to the reference builds; "
                                        "oracle/_ref lacks %s" % ", ".join(missing))
        self.data = {}
        if os.path.exists(self.PATH):
            with open(self.PATH) as f:
                self.data = json.load(f)

    @staticmethod
    def digest(**items):
        import hashlib
        import numpy as np
        out = {}
        for k, v in items.items():
            if isinstance(v, np.ndarray):
                v = np.ascontiguousarray(v).tobytes()
            if isinstance(v, str) and len(v) > 4096:
                v = v.encode()
            if isinstance(v, bytes):
                v = "sha256:" + hashlib.sha256(v).hexdigest()
            elif isinstance(v, np.integer):
                v = int(v)
            out[k] = v
        return out

    def check(self, key, got):
        if self.out:
            self.data[key] = got
            return
        assert key in self.data, "no stored output for %s" % key
        exp = self.data[key]
        assert got == exp, (key, {k: (got.get(k), exp.get(k)) for k in set(got) | set(exp) if got.get(k) != exp.get(k)})

    def save(self):
        import json
        with open(self.out, "w") as f:
            json.dump(self.data, f, indent=0, sort_keys=True)


_recorded = []


@pytest.fixture(scope="session")
def recorded():
    if not _recorded:
        _recorded.append(Recorded())
    return _recorded[0]


def pytest_sessionfinish(session, exitstatus):
    if _recorded and _recorded[0].out and exitstatus == 0:
        _recorded[0].save()


@pytest.fixture(scope="session")
def golden():
    import json
    import numpy as np
    here = os.path.join(ROOT, "tests", "golden")
    with open(os.path.join(here, "golden_stats.json")) as f:
        stats = json.load(f)
    ues = dict(np.load(os.path.join(here, "golden_ues.npz")))
    return stats, ues
