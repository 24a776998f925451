"""CPU: host-side mirror of the reference API — module tree, nethook surgery, DataBag, z
sampling, mask decoding, cache format, paste/crop helpers, and that the C-ABI library loads
and exports every declared symbol (no kernels are launched here)."""
import os
import re

import numpy as np
import pytest
import torch

from rewriting_b200 import _cabi
from rewriting_b200.utils import nethook, renormalize, runningstats, tally, zdataset
from rewriting_b200.utils.stylegan2 import models as sg2
from rewriting_b200.rewrite import ganrewrite
from conftest import ROOT


def test_cabi_loads_and_exports_every_declared_symbol():
    lib = _cabi.load()
    assert lib.rw_version() >= 100
    header = open(os.path.join(ROOT, 'include', 'rewriting_b200.h')).read()
    body = header[header.index('extern "C"'):]
    declared = set(re.findall(r'^(?:int|size_t|const char\*)\s+(rw_[a-z0-9_]+)\s*\(', body, re.M))
    assert declared, 'no declarations parsed'
    for name in sorted(declared):
        assert hasattr(lib, name), 'missing export ' + name
        assert name in _cabi.SIGNATURES, 'no ctypes prototype for ' + name
    assert lib.rw_gram_workspace_bytes(512, 512, 10890, 1) > 0


def test_ops_refuse_cpu_tensors():
    from rewriting_b200 import ops
    with pytest.raises(_cabi.RwError):
        ops.prep_keys(torch.zeros(1, 64, 4, 4))
    with pytest.raises(RuntimeError):
        runningstats.RunningSecondMoment().add(torch.zeros(8, 128))


def test_databag_semantics():
    d = sg2.DataBag(latent=torch.zeros(1), fmap=torch.ones(2))
    e = sg2.DataBag(d, fmap=torch.zeros(3))
    assert e.fmap.shape == (3,) and d.fmap.shape == (2,)      # copy-on-construct
    assert e.latent is d.latent
    e.output = torch.ones(1)
    assert 'output' in e and 'output' not in d
    assert e.get('noise', None) is None
    rebuilt = type(e)({k: v.detach() for k, v in e.items()})   # ganrewrite.py:708-729 idiom
    assert isinstance(rebuilt, sg2.DataBag) and set(rebuilt) == set(e)
    del e.output
    assert 'output' not in e
    with pytest.raises(AttributeError):
        _ = e.missing


def test_module_tree_and_state_dict_keys(seeded_model):
    sd = seeded_model.state_dict()
    assert len(sd) == 136
    assert sd['layer8.sconv.mconv.dconv.weight'].shape == (1, 512, 512, 3, 3)
    assert sd['layer2.conv.mconv.dconv.weight'].shape == (1, 512, 512, 3, 3)
    assert sd['layer13.sconv.mconv.dconv.weight'].shape == (1, 128, 256, 3, 3)
    assert sd['layer13.sconv.mconv.blur.kernel'].shape == (4, 4)
    assert sd['to_rgb7.rgb.conv.weight'].shape == (1, 3, 128, 1, 1)
    assert sd['latents.latent_avg'].ndim == 0
    assert sd['noises.noise_12'].shape == (1, 1, 256, 256)
    assert sum(p.numel() for p in seeded_model.parameters()) == 30034338
    names = [n for n, _ in seeded_model.named_children()]
    assert names[:7] == ['bag_in', 'style', 'latents', 'noises', 'input', 'layer2', 'to_rgb1']
    assert names[-1] == 'output'


def test_subsequence_split_matches_reference_structure(seeded_model):
    first, last = 'layer8.sconv.mconv.dconv', 'layer8.sconv.activate'
    ctx = nethook.subsequence(seeded_model, upto_layer=first, share_weights=True)
    tgt = nethook.subsequence(seeded_model, first_layer=first, last_layer=last,
                              share_weights=True)
    rnd = nethook.subsequence(seeded_model, after_layer=last, share_weights=True)
    leaf = lambda m: [n for n, c in m.named_modules() if len(list(c.children())) == 0]
    assert [n for n, _ in ctx.named_children()][-1] == 'layer8'
    assert [n for n, _ in ctx.layer8.named_children()] == ['lat6', 'sconv']
    assert [n for n, _ in ctx.layer8.sconv.mconv.named_children()] == ['modulation', 'adain']
    assert leaf(tgt) == ['layer8.sconv.mconv.dconv', 'layer8.sconv.noise', 'layer8.sconv.activate']
    assert [n for n, _ in rnd.named_children()][:3] == ['to_rgb4', 'up_rgb4', 'layer9']
    # whole children are the original objects, entered levels are plain Sequentials
    assert ctx.layer7 is seeded_model.layer7
    assert type(tgt.layer8.sconv) is torch.nn.Sequential
    assert tgt.layer8.sconv.mconv.dconv is seeded_model.layer8.sconv.mconv.dconv
    n = lambda m: len(m.state_dict())
    assert n(ctx) + n(tgt) + n(rnd) == 136
    with pytest.raises(ValueError):
        nethook.subsequence(seeded_model, first_layer='layer99')
    one = nethook.subsequence(seeded_model, single_layer='layer4', share_weights=False)
    assert one.layer4 is not seeded_model.layer4


def test_instrumented_model_hooks_and_unhooks():
    net = torch.nn.Sequential()
    net.add_module('a', torch.nn.Linear(4, 4))
    net.add_module('b', torch.nn.ReLU())
    x = torch.randn(2, 4)
    with nethook.InstrumentedModel(net) as inst:
        inst.retain_layer('a')
        inst.edit_layer('b', ablation=1.0, replacement=torch.zeros(4))
        y = inst(x)
        assert torch.equal(y, torch.zeros(2, 4))
        assert torch.allclose(inst.retained_layer('a'), net.a(x))
        assert 'forward' in net.a.__dict__
        only_a = inst(x, layer='a')
        assert torch.allclose(only_a, net.a(x))
    assert 'forward' not in net.a.__dict__ and 'forward' not in net.__dict__
    assert (net(x) >= 0).all()


def test_z_samples_are_prefix_stable():
    a = zdataset.standard_z_sample(5, 512, seed=1)
    b = zdataset.standard_z_sample(50, 512, seed=1)
    assert a.dtype == torch.float32 and torch.equal(a, b[:5])
    ref = np.random.RandomState(1).standard_normal(5 * 512).reshape(5, 512).astype('float32')
    assert np.array_equal(a.numpy(), ref)


def test_mask_decoding_uses_red_channel(edit_request):
    url = edit_request['object'][1]
    area = renormalize.from_url(url, target='pt', size=(32, 32))[0]
    assert area.shape == (32, 32) and 0 < float(area.sum()) < 32 * 32
    assert float(area.max()) == 1.0 and float(area.min()) == 0.0
    full = renormalize.from_url(url, target='pt')
    assert full.shape == (3, 256, 256)
    t, l, b, r = ganrewrite.positive_bounding_box(area)
    assert 0 <= t < b <= 32 and 0 <= l < r <= 32
    assert ganrewrite.positive_bounding_box(torch.zeros(4, 4)) == (0, 0, 0, 0)


def test_paste_and_crop_helpers():
    src = torch.zeros(1, 2, 8, 8)
    clip = torch.ones(1, 2, 3, 3)
    out, (t, l, b, r) = ganrewrite.paste_clip_at_center(src, clip, (7, 0))
    assert (t, l, b, r) == (5, 0, 8, 3) and out[0, 0, 5:8, 0:3].sum() == 9 and out.sum() == 18
    half = torch.full((3, 3), 0.5)
    out2, _ = ganrewrite.paste_clip_at_center(src + 2, clip, (4, 4), half)
    assert torch.allclose(out2[0, 0, 3:6, 3:6], torch.full((3, 3), 1.5))
    s, tg, sb, tb = ganrewrite.crop_clip_to_bounds(torch.zeros(1, 1, 4, 4), torch.zeros(1, 1, 8, 8),
                                                   (1, 2, 5, 7))
    assert sb == (0, 1, 3, 4) and tb == (0, 2, 6, 8)
    assert s.shape[2:] == (3, 3) and tg.shape[2:] == (6, 6)


def test_second_moment_cache_format_roundtrip(tmp_path):
    r = runningstats.RunningSecondMoment()
    r.count, r.mom2 = 256000, torch.eye(8) * 3
    path = str(tmp_path / 'cache' / 'r2m.npz')
    tally.save_cached_state(path, r, dict(sample_size=None))
    dat = np.load(path, allow_pickle=True)
    assert set(dat.files) == {'constructor', 'count', 'mom2', 'sample_size'}
    assert str(dat['constructor']).endswith('runningstats.RunningSecondMoment()')
    assert dat['mom2'].dtype == np.float32
    back = tally.load_cached_state(path, dict(sample_size=None))
    r2 = runningstats.RunningSecondMoment(state=back)
    assert r2.count == 256000 and torch.equal(r2.moment(), torch.eye(8) * 3 / 256000)
    assert tally.load_cached_state(path, dict(sample_size=7)) is None    # args changed
    # tally_second_moment returns the cached object without calling compute
    out = tally.tally_second_moment(lambda z: 1 / 0, torch.zeros(4, 2), cachefile=path)
    assert out.count == 256000


def test_zca_from_cov_whitens():
    torch.manual_seed(0)
    a = torch.randn(4000, 16) @ torch.randn(16, 16)
    C = a.t() @ a / 4000
    Z = ganrewrite.zca_from_cov(C)
    assert torch.allclose(Z @ C @ Z, torch.eye(16), atol=2e-3)
    assert torch.allclose(Z, Z.t(), atol=1e-5)


def test_checkpoint_key_conversion_from_rosinality_names(seeded_model):
    sd = seeded_model.state_dict()

    def back(k):   # inverse of the loader's renaming, for the keys it handles
        k = re.sub(r'^layer2\.conv\.mconv\.dconv\.weight$', 'conv1.conv.weight', k)
        k = re.sub(r'^layer2\.conv\.mconv\.', 'conv1.conv.', k)
        k = re.sub(r'^layer2\.conv\.', 'conv1.', k)
        m = re.match(r'^layer(\d+)\.sconv\.mconv\.dconv\.weight$', k)
        if m:
            return 'convs.%d.conv.weight' % (int(m.group(1)) - 3)
        k = re.sub(r'^layer(\d+)\.sconv\.mconv\.', lambda m: 'convs.%d.conv.' % (int(m.group(1)) - 3), k)
        k = re.sub(r'^layer(\d+)\.sconv\.', lambda m: 'convs.%d.' % (int(m.group(1)) - 3), k)
        k = re.sub(r'^to_rgb1\.rgb\.', 'to_rgb1.', k)
        k = re.sub(r'^up_rgb(\d+)\.', lambda m: 'to_rgbs.%d.upsample.' % (int(m.group(1)) - 1), k)
        k = re.sub(r'^to_rgb(\d+)\.rgb\.', lambda m: 'to_rgbs.%d.' % (int(m.group(1)) - 2), k)
        return k
    ros = {back(k): v for k, v in sd.items() if not k.startswith(('noises', 'latents'))}
    fresh = sg2.SeqStyleGAN2(256, 512, 8, mconv='seq')
    fresh.load_state_dict({'g_ema': ros, 'latent_avg': torch.zeros(512)})
    got = fresh.state_dict()
    for k in sd:
        if k == 'latents.latent_avg' or k.startswith('noises'):
            continue
        assert torch.equal(got[k], sd[k]), k
    # reference-compatible default: the buffer stays 0-dim (no truncation, same images as the
    # reference for a given z); real_truncation=True is the explicit opt-in
    assert got['latents.latent_avg'].ndim == 0
    opt = sg2.SeqStyleGAN2(256, 512, 8, mconv='seq', truncation=0.5, real_truncation=True)
    opt.load_state_dict({'g_ema': ros, 'latent_avg': torch.arange(512.)})
    assert opt.state_dict()['latents.latent_avg'].shape == (512,)
    w = torch.randn(3, 512)
    lat = opt.latents(sg2.DataBag(latent=w)).latent
    assert torch.allclose(lat[:, 0], torch.arange(512.) + 0.5 * (w - torch.arange(512.)))
    keep = sg2.SeqStyleGAN2(256, 512, 8, mconv='seq', truncation=0.5)
    keep.load_state_dict({'g_ema': ros, 'latent_avg': torch.arange(512.)})
    assert torch.equal(keep.latents(sg2.DataBag(latent=w)).latent[:, 0], w)


def test_shard_range_partitions_exactly():
    from rewriting_b200 import dist as rdist
    for n in (0, 1, 7, 16, 50010):
        for R in (1, 2, 3, 8):
            spans = [rdist.shard_range(n, r, R) for r in range(R)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))          # contiguous
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1 and sum(sizes) == n


def test_install_aliases_serves_the_reference_ui_over_this_rewriter(tmp_path):
    """`from rewrite import ganrewrite, rewriteapp` in a notebook: this package's rewriter and
    overlay renderer, the reference's device-independent GanRewriteApp / widgets.  The checkout
    is a stand-in holding only the module names this package does not provide."""
    import subprocess
    import sys
    ref = tmp_path / 'reference'
    for sub, mod, body in (('rewrite', 'rewriteapp', 'class GanRewriteApp(object):\n    pass\n'),
                           ('rewrite', 'ganrewrite', 'raise ImportError("shadowed")\n'),
                           ('utils', 'labwidget', 'class Widget(object):\n    pass\n'),
                           ('utils', 'imgviz', 'raise ImportError("shadowed")\n')):
        (ref / sub).mkdir(parents=True, exist_ok=True)
        (ref / sub / '__init__.py').write_text('')
        (ref / sub / (mod + '.py')).write_text(body)
    code = '''
import sys, types
sys.path.insert(0, %r)
if 'IPython' not in sys.modules:
    try:
        import IPython
    except ImportError:
        m = types.ModuleType('IPython'); d = types.ModuleType('IPython.display')
        d.display = lambda *a, **k: None; m.display = d
        sys.modules['IPython'] = m; sys.modules['IPython.display'] = d
import rewriting_b200
rewriting_b200.install_aliases(%r)
from rewrite import ganrewrite, rewriteapp
from utils import imgviz, labwidget, runningstats
assert ganrewrite.__file__.startswith(%r), ganrewrite.__file__
assert imgviz.__file__.startswith(%r) and runningstats.__file__.startswith(%r)
assert rewriteapp.__file__.startswith(%r) and labwidget.__file__.startswith(%r)
assert hasattr(rewriteapp, 'GanRewriteApp') and hasattr(ganrewrite, 'SeqStyleGanRewriter')
print('ok')
''' % (ROOT, str(ref), ROOT, ROOT, ROOT, str(ref), str(ref))
    r = subprocess.run([sys.executable, '-W', 'ignore', '-c', code], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith('ok'), r.stderr[-2000:]


def test_frechet_statistics_match_the_scipy_formula():
    """sampling.frechet_distance / activation_statistics vs the reference's numpy + scipy
    formula (metrics/fid.py:137-175: sqrtm of the covariance product)."""
    import numpy as np
    from scipy import linalg
    from rewriting_b200 import sampling
    rng = np.random.RandomState(0)
    a = rng.randn(500, 24) @ rng.randn(24, 24)
    b = rng.randn(400, 24) @ rng.randn(24, 24) + 0.3
    mu1, s1 = sampling.activation_statistics(torch.from_numpy(a))
    mu2, s2 = sampling.activation_statistics(torch.from_numpy(b))
    np.testing.assert_allclose(s1.numpy(), np.cov(a, rowvar=False), rtol=1e-10, atol=1e-12)
    covmean = linalg.sqrtm(np.cov(a, rowvar=False).dot(np.cov(b, rowvar=False)))
    diff = a.mean(0) - b.mean(0)
    want = diff.dot(diff) + np.trace(np.cov(a, rowvar=False)) + np.trace(np.cov(b, rowvar=False)) \
        - 2 * np.trace(covmean.real)
    got = sampling.frechet_distance(mu1, s1, mu2, s2)
    assert abs(got - want) < 1e-6 * max(1.0, abs(want))
    img = torch.rand(2, 3, 4, 4) * 2 - 1
    f = sampling.pt_to_float255_nhwc(img)
    assert f.shape == (2, 4, 4, 3) and float(f.min()) >= 0 and float(f.max()) <= 255
    assert torch.allclose(f[0, 1, 2], ((img[0, :, 1, 2] / 2 + 0.5) * 255))


def test_seeded_vgg16_is_deterministic_and_leaves_the_rng_alone():
    """The stand-in for the pretrained perceptual network of all_weights_insert (tests, goldens):
    same weights on every call and machine, global RNG state untouched."""
    from rewriting_b200.synthetic import seeded_vgg16
    torch.manual_seed(123)
    before = torch.random.get_rng_state().clone()
    a = seeded_vgg16()
    assert torch.equal(torch.random.get_rng_state(), before)
    b = seeded_vgg16()
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
    assert len(list(a.features.children())) == 31 and not a.training
    assert not torch.equal(seeded_vgg16(seed=1).features[0].weight, a.features[0].weight)


def test_up_fused_eligibility_matches_the_kernel_limits(monkeypatch):
    """Shapes the one-kernel upsampling StyledConv takes (csrc/upconv_tc.cu: power-of-two square
    inputs of width 4..128, Cin % 64 == 0, Cout % 16 == 0, rank-one 4x4 FIR); everything else —
    and RW_UP_FUSED=0 — keeps the conv_transpose + blur pair."""
    from rewriting_b200 import ops
    k1 = torch.tensor([1., 3., 3., 1.])
    sep = k1[:, None] * k1[None, :] / 16
    assert ops.up_fused_eligible(512, 512, 4, 4, sep)
    assert ops.up_fused_eligible(256, 128, 128, 128, sep)
    assert not ops.up_fused_eligible(256, 128, 256, 256, sep)       # wider than a tile
    assert not ops.up_fused_eligible(256, 128, 24, 24, sep)         # not a power of two
    assert not ops.up_fused_eligible(256, 128, 32, 64, sep)         # not square
    assert not ops.up_fused_eligible(96, 128, 32, 32, sep)          # Cin % 64
    assert not ops.up_fused_eligible(128, 24, 32, 32, sep)          # Cout % 16
    nonsep = sep.clone()
    nonsep[1, 2] += 0.01
    assert not ops.up_fused_eligible(128, 32, 32, 32, nonsep)       # FIR not rank one
    monkeypatch.setenv('RW_UP_FUSED', '0')
    assert not ops.up_fused_eligible(512, 512, 4, 4, sep)
