"""CPU: the oracle and this repo's constructors at 512^2 and 1024^2 against the goldens pinned from
the reference (oracle/make_golden_highres.py)."""
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import sg2_oracle as orc
from conftest import GOLD


@pytest.fixture(scope='module')
def hgold():
    return dict(np.load(os.path.join(GOLD, 'sg2_highres.npz')))


def _seeded(size):
    from rewriting_b200.utils.stylegan2 import SeqStyleGAN2
    return orc.seeded_state_dict(lambda: SeqStyleGAN2(size, style_dim=512, n_mlp=8, mconv='seq'))


@pytest.mark.parametrize('size', [512, 1024])
def test_seeded_constructor_checksums(size):
    with open(os.path.join(GOLD, 'weights_checksum_highres.json')) as f:
        want = json.load(f)[str(size)]
    sd = _seeded(size).state_dict()
    assert list(sd.keys()) == list(want.keys())
    for k, v in sd.items():
        assert [float(v.double().sum()), float(v.double().abs().sum())] == want[k], k


def test_oracle_512_pixels_bit_exact(z40, hgold):
    sd = {k: v.clone() for k, v in _seeded(512).state_dict().items()}
    with torch.no_grad():
        pix = orc.generator_forward(sd, z40[:2], size=512)
    assert np.array_equal(pix[:, :, ::16, ::16].numpy(), hgold['pix512_sub'])
    np.testing.assert_array_equal(pix.double().sum(dim=(2, 3)).numpy(), hgold['pix512_sum'])


def test_oracle_insert_loop_reproduces_smile_edit(hgold):
    """The oracle's rewrite loop on the 1024^2 generator's layer 10 (goal crops from the golden):
    the rank-one update Lambda d^T and the loss trajectory of the reference's 50 iterations."""
    layer = int(hgold['layer'])
    sd = _seeded(1024).state_dict()
    p = orc._layer_params(sd, 'layer%d' % layer)
    d = torch.from_numpy(hgold['smile_d'])
    losses = []
    W = orc.insert_loop(p['weight'], torch.from_numpy(hgold['smile_goal_in_fmap']),
                        torch.from_numpy(hgold['smile_goal_in_style']),
                        torch.from_numpy(hgold['smile_goal_out_fmap']), p['noise_w'], p['bias'], d,
                        int(hgold['niter']), piter=10, lr=0.05, record_loss=losses)
    lam = torch.from_numpy(hgold['smile_lambda']).double()
    dW_gold = lam[:, None] * d.double()[0][None, :, None, None]
    err = ((W - p['weight'])[0].double() - dW_gold).abs().max().item()
    assert err < 1e-4 * max(1.0, dW_gold.abs().max().item()), err
    np.testing.assert_allclose(np.array(losses), hgold['smile_losses'], rtol=1e-5)
    assert math.isfinite(losses[-1]) and losses[-1] < losses[0]
