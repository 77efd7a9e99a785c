"""Stored answers of the reference comparisons (tests/golden/reference_answers.json).

The tests that hold the oracle and the host layer against the reference's own code (oracle/_ref, built from a
reference checkout named by DDC_REFERENCE_DIR) draw seeded cases.  On every case the reference's answer had to
equal this repository's answer; the file stores a digest of that answer, case by case, so the comparison also runs
where no reference checkout exists.  Where oracle/_ref is built the live comparison runs as well.

    DDC_RECORD_REFERENCE_ANSWERS=1 python -m pytest tests/test_reference_hostpath.py tests/test_oracle_golden.py \
        tests/test_host_layer_cpu.py -m "not gpu"

re-records the digests; each entry notes whether the live comparison with the reference's code ran while it was
recorded ("checked_against_reference_code")."""
import hashlib
import json
import os

import numpy as np

from conftest import ROOT

PATH = os.path.join(ROOT, "tests", "golden", "reference_answers.json")
RECORD = bool(os.environ.get("DDC_RECORD_REFERENCE_ANSWERS"))


def _canon(x):
    if isinstance(x, np.ndarray):
        return _canon(x.tolist())
    if isinstance(x, np.generic):
        return x.item()
    if isinstance(x, dict):
        items = [[_canon(k), _canon(v)] for k, v in x.items()]
        return sorted(items, key=lambda kv: json.dumps(kv[0]))
    if isinstance(x, (list, tuple)):
        return [_canon(v) for v in x]
    return x


def digest(x) -> str:
    return hashlib.sha256(json.dumps(_canon(x), separators=(",", ":")).encode()).hexdigest()[:20]


class Answers:
    """the stored answers of one test: check() one case after another, then finish()"""

    def __init__(self, test: str, live: bool):
        self.test, self.live, self.got = test, live, []
        with open(PATH) as f:
            self.want = json.load(f)["answers"].get(test, {}).get("digests")
        assert RECORD or self.want is not None, "no stored answers for %s" % test

    def check(self, answer, ctx=None):
        d = digest(answer)
        if not RECORD:
            i = len(self.got)
            assert i < len(self.want), (self.test, "more cases than stored answers")
            assert d == self.want[i], (self.test, "case %d differs from the stored answer" % i, ctx)
        self.got.append(d)

    def finish(self):
        if not RECORD:
            assert len(self.got) == len(self.want), (self.test, len(self.got), len(self.want))
            return
        with open(PATH) as f:
            data = json.load(f)
        data["answers"][self.test] = {"checked_against_reference_code": self.live, "digests": self.got}
        with open(PATH, "w") as f:
            json.dump(data, f, indent=1, sort_keys=True)
            f.write("\n")
