"""TEST INFRASTRUCTURE ONLY — the device-independent host helpers (zdataset, renormalize, the
rewriter's crop / paste geometry, zca_from_cov, nethook subsequence / InstrumentedModel,
FixedSubsetSampler) run on seeded inputs, for either implementation.

`cases(ns)` takes a namespace with `zdataset`, `renormalize`, `ganrewrite`, `nethook` and
`FixedSubsetSampler` and returns {check name: list of outputs}.  oracle/make_golden_host.py runs
it on the live reference and stores the answers in tests/golden/host_helpers.npz;
tests/test_host_vs_reference.py runs it on this package and requires every output to be
bit-identical to the stored one.  The inputs are regenerated from the seeds on both sides.
"""
from collections import OrderedDict

import numpy as np
import torch

RENORM_KINDS = ('zc', 'pt', 'imagenet', 'byte')
FROM_URL = [('zc', None), ('pt', (32, 32)), ('byte', (16, 24))]
SUBSEQUENCES = [dict(first_layer='b.b2', last_layer='c'), dict(after_layer='a', upto_layer='b.b3'),
                dict(first_layer='b', last_layer='b'), dict(upto_layer='b.b2'),
                dict(after_layer='b.b1')]


def toy():
    torch.manual_seed(3)
    return torch.nn.Sequential(OrderedDict([
        ('a', torch.nn.Linear(6, 6)),
        ('b', torch.nn.Sequential(OrderedDict([('b1', torch.nn.Linear(6, 6)), ('b2', torch.nn.Tanh()),
                                               ('b3', torch.nn.Linear(6, 6))]))),
        ('c', torch.nn.ReLU()), ('d', torch.nn.Linear(6, 3))]))


def _sample(a, n=64):
    """[shape, n elements at fixed seeded positions] of a larger output: keeps the stored
    answers small while a misplaced window or a wrong per-channel constant still shows."""
    a = np.asarray(a.detach().cpu() if isinstance(a, torch.Tensor) else a)
    idx = np.sort(np.random.RandomState(a.size).choice(a.size, min(n, a.size), replace=False))
    return [np.array(a.shape), a.reshape(-1)[idx]]


def _np(a):
    if isinstance(a, torch.Tensor):
        return a.detach().cpu().numpy()
    return np.asarray(a)


def cases(ns, url=None):
    """Outputs of `ns`'s helpers.  `url` replaces the as_url() string fed to from_url(), so that
    both implementations decode the same bytes."""
    out = OrderedDict()
    rng = np.random.RandomState(0)
    g = torch.Generator().manual_seed(0)

    out['z_sample'] = [ns.zdataset.standard_z_sample(n, d, seed=s)
                       for n, d, s in [(5, 512, 1), (37, 64, 10), (1, 512, 20)]]
    out['y_sample'] = [ns.zdataset.standard_y_sample(50, 10, seed=3)]

    img = torch.rand(3, 40, 52, generator=g) * 2 - 1
    conv = []
    for src in RENORM_KINDS:
        x = (img if src == 'zc' else ns.renormalize.as_tensor(img, 'zc', src)).float()
        for tgt in RENORM_KINDS:
            conv += _sample(ns.renormalize.as_tensor(x, src, tgt).float(), 256)
    out['renorm_as_tensor'] = conv
    out['renorm_as_image'] = [np.asarray(ns.renormalize.as_image(img))]
    mine_url = ns.renormalize.as_url(img)
    out['renorm_url'] = [np.array(mine_url)]
    url = url or mine_url
    out['renorm_from_url'] = sum((_sample(ns.renormalize.from_url(url, target=t, size=sz), 256)
                                  for t, sz in FROM_URL), [])

    geom = {k: [] for k in ('bbox', 'center', 'paste', 'crop')}
    for trial in range(25):
        h, w = int(rng.randint(6, 40)), int(rng.randint(6, 40))
        mask = torch.zeros(h, w)
        t, l = int(rng.randint(0, h - 2)), int(rng.randint(0, w - 2))
        b, r = int(rng.randint(t + 1, h + 1)), int(rng.randint(l + 1, w + 1))
        mask[t:b, l:r] = torch.rand(b - t, r - l, generator=g) + 0.01
        geom['bbox'].append(ns.ganrewrite.positive_bounding_box(mask))
        geom['center'].append(ns.ganrewrite.centered_location(mask))
        src = torch.randn(1, 4, h, w, generator=g)
        ch, cw = int(rng.randint(1, h + 1)), int(rng.randint(1, w + 1))
        clip = torch.randn(1, 4, ch, cw, generator=g)
        area = torch.rand(ch, cw, generator=g)
        center = (int(rng.randint(0, h)), int(rng.randint(0, w)))
        for ar in (None, area):
            # the pasted window, its bounds, and whether everything outside it is `src`
            pasted, (pt, pl, pb, pr) = ns.ganrewrite.paste_clip_at_center(src, clip, center, ar)
            outside = torch.ones_like(src, dtype=torch.bool)
            outside[:, :, pt:pb, pl:pr] = False
            geom['paste'] += _sample(pasted[:, :, pt:pb, pl:pr]) + [
                (pt, pl, pb, pr), bool(torch.equal(pasted[outside], src[outside]))]
        tgt = torch.randn(1, 4, 2 * h, 2 * w, generator=g)
        cs, ct, sb, tb = ns.ganrewrite.crop_clip_to_bounds(src, tgt, (t, l, b, r))
        geom['crop'] += _sample(cs) + _sample(ct) + [sb, tb]
    out.update(('geom_' + k, v) for k, v in geom.items())

    a = torch.randn(200, 24, generator=g)
    out['zca_from_cov'] = [ns.ganrewrite.zca_from_cov(a.t() @ a / 200)]

    x = torch.randn(5, 6, generator=g)
    outs, names = [], []
    for kw in SUBSEQUENCES:
        s = ns.nethook.subsequence(toy(), share_weights=True, **kw)
        outs.append(s(x))
        names.append(np.array([n for n, _ in s.named_modules()]))
    out['subsequence_output'] = outs
    out['subsequence_names'] = names

    im = ns.nethook.InstrumentedModel(toy())
    im.retain_layers(['b.b1', ('d', 'out')])
    y = im(x)
    out['imodel_retained'] = [im.retained_layer('b.b1'), im.retained_layer('out'), y]
    im.edit_layer('b.b1', ablation=0.5, replacement=torch.randn(5, 6, generator=g))
    out['imodel_edit'] = [im(x)]
    im.remove_edits()
    out['imodel_edits_removed'] = [im(x)]

    out['sampler'] = [np.array(list(ns.FixedSubsetSampler([3, 1, 4, 1, 5]))),
                      np.array(len(ns.FixedSubsetSampler(list(range(7)))))]
    return OrderedDict((k, [_np(a) for a in v]) for k, v in out.items())
