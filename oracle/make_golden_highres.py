"""TEST INFRASTRUCTURE ONLY — pins the 512^2 and 1024^2 StyleGAN2 generators against the live
reference and writes tests/golden/sg2_highres.npz and tests/golden/weights_checksum_highres.json.
Runs in the authoring container only (needs the read-only reference at /root/reference):

    python oracle/make_golden_highres.py

What is pinned (reference executed unmodified through oracle/ref_shim.py, seeded synthetic
weights as in make_golden.py):
  * SeqStyleGAN2(512) and SeqStyleGAN2(1024), mconv='seq', B=2: pixels, stored as a stride-16
    subsample plus full-image float64 sums (the oracle must match bit-exactly);
  * that this repo's constructors under the same seed give identical parameters (checksums);
  * the `smile` edit on the seeded 1024^2 generator: layer 10, rank 1,
    C from 40 z, 50 insert iterations -> d, Lambda of the rank-one update dW = Lambda d^T
    (not the 9.4 MB weight), goal crops, loss trajectory, pixels of the edited generator.

tests/golden/smile.json is the reference's notebooks/masks/stylegan/celebhq/smile.json, copied
unchanged (a UI edit request of the reference's face experiments; reference data, not code).
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, 'tests', 'golden')

from oracle import sg2_oracle as orc          # noqa: E402
from oracle.ref_shim import load_reference    # noqa: E402

N_Z = 40
LAYER = 10
NITER = 50
SIZES = (512, 1024)
SUB = 16


def checksum(sd):
    return {k: [float(v.double().sum()), float(v.double().abs().sum())] for k, v in sd.items()}


def pixel_stats(pix):
    """[B,3,S,S] -> (stride-16 subsample, per-(b,c) float64 sum and abs-sum)"""
    p64 = pix.double()
    return (pix[:, :, ::SUB, ::SUB].numpy(), p64.sum(dim=(2, 3)).numpy(),
            p64.abs().sum(dim=(2, 3)).numpy())


def seeded(ctor_mod, size):
    return orc.seeded_state_dict(
        lambda: ctor_mod.SeqStyleGAN2(size, style_dim=512, n_mlp=8, mconv='seq')).eval()


def main():
    torch.set_num_threads(os.cpu_count())
    ref = load_reference()
    from rewriting_b200.utils import stylegan2 as mine_mod
    z = ref.zdataset.standard_z_sample(N_Z, 512, seed=1)
    out = {'n_z': N_Z, 'layer': LAYER, 'niter': NITER, 'sub': SUB}
    sums = {}
    models = {}
    for size in SIZES:
        ref_model = seeded(ref.models, size)
        sd = {k: v.clone() for k, v in ref_model.state_dict().items()}
        my_sd = seeded(mine_mod, size).state_dict()
        assert list(my_sd.keys()) == list(sd.keys()), 'state_dict keys differ at %d' % size
        for k in sd:
            assert torch.equal(my_sd[k], sd[k]), 'seeded init differs at %s (%d)' % (k, size)
        sums[str(size)] = checksum(sd)
        with torch.no_grad():
            pix_ref = ref_model(z[:2])
            pix_orc = orc.generator_forward(sd, z[:2], size=size)
        assert torch.equal(pix_ref, pix_orc), 'oracle differs from the reference at %d: %g' % (
            size, (pix_ref - pix_orc).abs().max())
        print('%d: seeded init identical (%d tensors), oracle pixels bit-exact, range %.2f..%.2f'
              % (size, len(sd), pix_ref.min(), pix_ref.max()))
        s, su, sa = pixel_stats(pix_ref)
        out['pix%d_sub' % size], out['pix%d_sum' % size], out['pix%d_abssum' % size] = s, su, sa
        models[size] = ref_model

    # ---- the smile edit on the 1024^2 generator (experiments: faces, smile.json, layer 10) ----
    with open(os.path.join(GOLD, 'smile.json')) as f:
        request = json.load(f)
    model = models[1024]
    zds = torch.utils.data.TensorDataset(z)
    gw = ref.ganrewrite.SeqStyleGanRewriter(model, zds, LAYER, cachedir=None)
    with torch.no_grad():
        obj_acts, _, obj_area, _ = gw.object_from_selection(*request['object'])
        goal_in, goal_out, _, _ = gw.paste_from_selection(request['paste'][0], request['paste'][1],
                                                          obj_acts, obj_area)
        key_examples = request.get('key', [request['paste']])
        d = gw.multi_key_from_selection(key_examples, rank=1)
    W0 = gw.target_weights().detach().clone()
    losses = []
    gw.insert(goal_in, goal_out, d, niter=NITER, piter=10, lr=0.05,
              update_callback=lambda it, loss: losses.append(float(loss)))
    W1 = gw.target_weights().detach().clone()
    dW = (W1 - W0)[0].double()                                   # [Cout, Cin, 3, 3]
    dd = d.double()[0]
    lam = torch.einsum('oiyx,i->oyx', dW, dd) / dd.dot(dd)       # dW = Lambda d^T
    resid = (dW - lam[:, None] * dd[None, :, None, None]).abs().max().item()
    print('smile: %d goal pixels, loss %.4g -> %.4g, |dW|max %.3g, rank-one residual %.3g' % (
        goal_in.fmap.shape[-1] * goal_in.fmap.shape[-2], losses[0], losses[-1],
        dW.abs().max().item(), resid))
    assert resid < 1e-6 * max(1.0, dW.abs().max().item())
    with torch.no_grad():
        pix_edit = model(z[:2])
    s, su, sa = pixel_stats(pix_edit)
    out.update(
        smile_d=d.numpy(), smile_lambda=lam.float().numpy(), smile_w0_sub=W0[0, ::37, ::41].numpy(),
        smile_goal_in_fmap=goal_in.fmap.numpy(), smile_goal_in_style=goal_in.style.numpy(),
        smile_goal_out_fmap=goal_out.fmap.numpy(),
        smile_losses=np.array(losses, dtype=np.float64),
        smile_pix_sub=s, smile_pix_sum=su, smile_pix_abssum=sa)
    np.savez_compressed(os.path.join(GOLD, 'sg2_highres.npz'), **out)
    with open(os.path.join(GOLD, 'weights_checksum_highres.json'), 'w') as f:
        json.dump(sums, f)
    print('wrote fixtures to', GOLD)


if __name__ == '__main__':
    main()
