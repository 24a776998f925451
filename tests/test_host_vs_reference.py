"""CPU: the device-independent host helpers of this package (zdataset, renormalize, the
rewriter's crop / paste geometry, zca_from_cov, nethook subsequence / InstrumentedModel,
FixedSubsetSampler) against what the live reference returned on the same seeded inputs
(oracle/host_cases.py; answers stored by oracle/make_golden_host.py)."""
import os
import types

import numpy as np
import torch

from oracle import host_cases
from rewriting_b200.rewrite import ganrewrite
from rewriting_b200.utils import nethook, renormalize, zdataset
from rewriting_b200.utils.sampler import FixedSubsetSampler

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'host_helpers.npz')


def test_host_helpers_equal_the_live_reference():
    gold = np.load(GOLD)
    ns = types.SimpleNamespace(zdataset=zdataset, renormalize=renormalize, ganrewrite=ganrewrite,
                               nethook=nethook, FixedSubsetSampler=FixedSubsetSampler)
    with torch.random.fork_rng():
        res = host_cases.cases(ns, url=str(gold['renorm_url/0']))
    want = {}
    for key in gold.files:
        name, i = key.rsplit('/', 1)
        want.setdefault(name, {})[int(i)] = gold[key]
    assert set(res) == set(want)
    bad = []
    for name, outs in res.items():
        assert len(outs) == len(want[name]), name
        for i, got in enumerate(outs):
            ref = want[name][i]
            if got.dtype.kind in 'US' or ref.dtype.kind in 'US':
                same = got.shape == ref.shape and bool(np.all(got == ref))
            else:                                      # bit-identical after widening to float64
                same = got.shape == ref.shape and np.array_equal(got.astype(np.float64),
                                                                 ref.astype(np.float64))
            if not same:
                bad.append('%s[%d]' % (name, i))
    assert not bad, bad
    assert len(res) >= 17

    # this package's own guarantees, beyond the reference's: subsequences share the parent's
    # parameters, and InstrumentedModel.close() restores the wrapped model
    with torch.random.fork_rng():
        x = torch.randn(5, 6, generator=torch.Generator().manual_seed(1))
        for kw in host_cases.SUBSEQUENCES:
            m = host_cases.toy()
            ids = {id(p) for p in m.parameters()}
            s = nethook.subsequence(m, share_weights=True, **kw)
            assert all(id(p) in ids for p in s.parameters()), kw
        m = host_cases.toy()
        im = nethook.InstrumentedModel(m)
        im.retain_layers(['b.b1', ('d', 'out')])
        im.edit_layer('b.b1', ablation=0.5, replacement=torch.randn(5, 6))
        im(x)
        im.close()
        assert torch.equal(m(x), host_cases.toy()(x))
