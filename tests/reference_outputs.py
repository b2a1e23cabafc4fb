"""What the original watsor project's own code returns, for the tests that compare this repository with it.

The outputs were recorded by running that code and are stored in tests/golden/reference/<name>.json, so the
comparisons run without it.  Where a checkout of the original project is readable (WATSOR_REFERENCE, else its usual
location: oracle/reference_build.find_reference), the tests import it and compute the outputs live instead; with
WATSOR_RECORD=1 as well, the run rewrites the stored files.  Arrays are stored as their SHA-256, shape and dtype: an
equality test on a digest is the same test as on the array."""
import atexit
import hashlib
import json
import os

import numpy as np

from oracle.reference_build import find_reference

REFERENCE = find_reference()
_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference')


def canon(v):
    """`v` as JSON stores it: tuples become lists, numpy scalars Python numbers, arrays a digest."""
    if isinstance(v, np.ndarray):
        v = np.ascontiguousarray(v)
        return {'sha256': hashlib.sha256(v.tobytes()).hexdigest(), 'shape': list(v.shape), 'dtype': str(v.dtype)}
    if isinstance(v, (list, tuple)):
        return [canon(x) for x in v]
    if isinstance(v, dict):
        return {str(k): canon(x) for k, x in v.items()}
    if isinstance(v, np.generic):
        return v.item()
    return v


class Recorded:
    def __init__(self, name):
        self.path = os.path.join(_DIR, name + '.json')
        self.data = {}
        if os.path.isfile(self.path):
            with open(self.path) as f:
                self.data = json.load(f)
        self.recording = bool(REFERENCE) and os.environ.get('WATSOR_RECORD') == '1'
        if self.recording:
            atexit.register(self.save)

    def __call__(self, key, compute):
        """The original project's output for `key`: `compute()` when it is importable, else the stored record.  A live
        output must equal the stored one unless the run is recording."""
        if REFERENCE:
            live = canon(compute())
            if key in self.data and not self.recording:
                assert live == self.data[key], 'the original project no longer gives the output stored for %r in %s' \
                    % (key, self.path)
            self.data[key] = live
        assert key in self.data, 'no recorded reference output for %r in %s' % (key, self.path)
        return self.data[key]

    def save(self):
        os.makedirs(_DIR, exist_ok=True)
        with open(self.path, 'w') as f:
            json.dump(self.data, f, sort_keys=True, separators=(',', ':'))
            f.write('\n')
