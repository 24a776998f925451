"""TEST INFRASTRUCTURE ONLY — golden answers of the live reference's device-independent host
helpers on the seeded inputs of oracle/host_cases.py (needs a checkout of the reference):

    python oracle/make_golden_host.py      ->  tests/golden/host_helpers.npz

Only the reference's outputs are stored, as `<check>/<index>`; the test regenerates the inputs
from the same seeds.
"""
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import host_cases                  # noqa: E402
from oracle.ref_shim import load_reference    # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden', 'host_helpers.npz')


def main():
    ref = load_reference()
    from utils.sampler import FixedSubsetSampler
    ns = types.SimpleNamespace(zdataset=ref.zdataset, renormalize=ref.renormalize,
                               ganrewrite=ref.ganrewrite, nethook=ref.nethook,
                               FixedSubsetSampler=FixedSubsetSampler)
    res = host_cases.cases(ns)
    flat = {'%s/%d' % (k, i): a for k, v in res.items() for i, a in enumerate(v)}
    np.savez_compressed(OUT, **flat)
    print('%s: %d arrays, %d bytes' % (OUT, len(flat), os.path.getsize(OUT)))


if __name__ == '__main__':
    main()
