"""Generate tests/golden/*.npz by running the UNMODIFIED reference module
(/root/reference/cspn_pytorch/models/cspn.py) on seeded CPU inputs.

Run in the build container (where /root/reference exists):
    python tests/golden/make_golden.py
The GPU box has no /root/reference; it checks parity against these committed files.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402
from cspn_b200.synth import make_inputs  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


CASES = [
    # name, seed, B, C, H, W, gch, sparse, n_sample, prop_time, norm_type
    ('small_8sum',        1, 2, 1, 13, 17, 8,  'signed',    40, 5,  '8sum'),
    ('small_8sum_abs',    2, 2, 1, 13, 17, 8,  'signed',    40, 5,  '8sum_abs'),
    ('nosparse_8sum',     3, 1, 1, 9,  20, 8,  None,        0,  7,  '8sum'),
    ('c3_shared',         4, 2, 3, 11, 12, 8,  'bernoulli', 30, 4,  '8sum_abs'),
    ('gch12_extra',       5, 1, 1, 8,  8,  12, 'bernoulli', 10, 3,  '8sum'),
    ('iter1',             6, 1, 1, 6,  9,  8,  'bernoulli', 10, 1,  '8sum'),
    ('iter48_abs',        7, 1, 1, 24, 40, 8,  'bernoulli', 60, 48, '8sum_abs'),
    ('odd_w_8sum',        8, 1, 1, 10, 15, 8,  'bernoulli', 20, 6,  '8sum'),
    ('tiny_1x1',          9, 1, 1, 1,  1,  8,  None,        0,  3,  '8sum'),
    ('row_1xW',          10, 1, 1, 1,  12, 8,  'bernoulli', 4,  5,  '8sum_abs'),
    ('nyu_8sum',         11, 1, 1, 228, 304, 8, 'bernoulli', 500, 24, '8sum'),      # BASELINE cfg1
    ('nyu_8sum_abs',     12, 1, 1, 228, 304, 8, 'bernoulli', 500, 24, '8sum_abs'),
]


def main():
    assert ref_loader.available(), 'reference tree not mounted'
    index = []
    for (name, seed, B, C, H, W, gch, sparse, ns, n, norm) in CASES:
        guidance, blur, sp = make_inputs(seed, B, C, H, W, gch, sparse, ns)
        out = ref_loader.reference_forward(guidance, blur, sp, n, norm)
        big = H * W > 10000
        rec = dict(seed=seed, B=B, C=C, H=H, W=W, gch=gch, sparse=str(sparse), n_sample=ns,
                   prop_time=n, norm_type=norm, out=out.numpy())
        if not big:   # small cases carry their inputs too, so they do not depend on torch's RNG stream
            rec.update(guidance=guidance.numpy(), blur=blur.numpy())
            if sp is not None:
                rec['sparse_depth'] = sp.numpy()
        np.savez_compressed(os.path.join(HERE, name + '.npz'), **rec)
        index.append(name)
        print(f'{name}: out shape {tuple(out.shape)} finite={bool(torch.isfinite(out).all())} '
              f'absmax={float(out.abs().max()):.4f}')
    # zero-affinity NaN semantics (SURVEY Appendix B): all-zero guidance -> NaN everywhere
    guidance = torch.zeros(1, 8, 4, 5)
    blur = torch.ones(1, 1, 4, 5)
    out = ref_loader.reference_forward(guidance, blur, None, 2, '8sum')
    np.savez_compressed(os.path.join(HERE, 'zero_guidance_nan.npz'), guidance=guidance.numpy(),
                        blur=blur.numpy(), out=out.numpy(), prop_time=2, norm_type='8sum',
                        seed=0, B=1, C=1, H=4, W=5, gch=8, sparse='None', n_sample=0)
    print('zero_guidance_nan: all nan =', bool(torch.isnan(out).all()))
    special_cases()
    port_cases()


PORT_SHAPES = [(2, 3, 7, 9), (1, 1, 16, 33)]
PORT_NORMS = ['8sum', '8sum_abs']


def port_name(norm, shape):
    return f'{norm}_' + 'x'.join(map(str, shape))


def port_cases():
    """tests/golden/port/*.npz: the reference's output for the cases on which the torch-op port must agree with it bit for
    bit (6 steps, 9 guidance channels, signed sparse depth); inputs travel with the file."""
    os.makedirs(os.path.join(HERE, 'port'), exist_ok=True)
    for norm in PORT_NORMS:
        for shape in PORT_SHAPES:
            g, d, s = make_inputs(123, *shape, 9, 'signed', 20)
            out = ref_loader.reference_forward(g, d, s, 6, norm)
            np.savez_compressed(os.path.join(HERE, 'port', port_name(norm, shape) + '.npz'), guidance=g.numpy(),
                                blur=d.numpy(), sparse_depth=s.numpy(), out=out.numpy(), prop_time=6, norm_type=norm)
            print(f'port {port_name(norm, shape)}: absmax={float(out.abs().max()):.4f}')


def save_special(name, guidance, blur, sp, n, norm):
    """Cases built by hand (non-finite / degenerate affinities): inputs always travel with the file."""
    out = ref_loader.reference_forward(guidance, blur, sp, n, norm)
    rec = dict(guidance=guidance.numpy(), blur=blur.numpy(), out=out.numpy(), prop_time=n, norm_type=norm, seed=0,
               B=guidance.shape[0], C=blur.shape[1], H=guidance.shape[2], W=guidance.shape[3], gch=guidance.shape[1],
               sparse=str(None if sp is None else 'given'), n_sample=0)
    if sp is not None:
        rec['sparse_depth'] = sp.numpy()
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **rec)
    o = out.numpy()
    print(f'{name}: nan={int(np.isnan(o).sum())} inf={int(np.isinf(o).sum())} of {o.size}')


def special_cases():
    """Shapes with W % 4 == 0 (the TMA/cluster kernel accepts them) that pin the reference's IEEE behaviour of
    cspn.py:135-138 (a / sum|a|): 0/0, a zero patch whose NaN spreads one pixel per step, subnormal sums, +-inf."""
    # all-zero guidance on a cluster-eligible shape
    save_special('nan_zero_guidance_4x8', torch.zeros(1, 8, 4, 8), torch.ones(1, 1, 4, 8), None, 2, '8sum')
    # a zero patch: pixels whose 8 gathered affinities are all zero are NaN from step 1 on and poison one more ring of
    # neighbours per step.  Steps 1, 2, 3: the NaN front must sit exactly where the reference's does (also at column 0,
    # i.e. lane 0 of the first strip, which is 3 columns from the first NaN pixel)
    for n in (1, 2, 3):
        g, d, s = make_inputs(50 + n, 1, 1, 12, 16, 8, 'bernoulli', 10)
        g[0, :, 3:8, 2:7] = 0
        save_special(f'nan_zero_patch_12x16_n{n}', g, d, s, n, '8sum')
    g, d, s = make_inputs(54, 2, 1, 40, 132, 8, 'signed', 60)           # wider than one 128-column strip: two strips
    g[0, :, 10:14, 126:131] = 0                                          # NaN source next to the strip cut
    g[1, :, 0:3, 0:3] = 0                                                # and in the image corner
    save_special('nan_zero_patch_40x132_n6', g, d, s, 6, '8sum_abs')
    # subnormal affinities: sum|a| ~ 1e-40 is not zero, the quotient is an ordinary number (needs true division:
    # 1/sum overflows)
    g, d, s = make_inputs(55, 1, 1, 8, 8, 8, 'bernoulli', 6)
    g[0, :, 2:6, 2:6] *= 1e-39
    g[0, :, 0:3, 5:8] *= 1e-44
    save_special('subnormal_affinity_8x8', g, d, s, 4, '8sum')
    # huge affinities: sum|a| near FLT_MAX (1/sum is subnormal) and overflowing to +inf
    g, d, s = make_inputs(56, 1, 1, 8, 12, 8, 'bernoulli', 6)
    g[0, :, 1:4, 1:5] *= 3e37
    g[0, :, 5:8, 6:11] *= 2e38
    save_special('huge_affinity_8x12', g, d, s, 3, '8sum')
    # +-inf in the guidance
    g, d, s = make_inputs(57, 1, 1, 8, 12, 8, 'bernoulli', 6)
    g[0, 2, 3, 4] = float('inf')
    g[0, 6, 5, 9] = float('-inf')
    save_special('inf_guidance_8x12', g, d, s, 2, '8sum')
    save_special('inf_guidance_abs_8x12', g, d, s, 2, '8sum_abs')


if __name__ == '__main__':
    main()
