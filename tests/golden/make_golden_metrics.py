"""Goldens for the device-side metrics / loss (cspn_b200/csrc/metrics.cu): outputs of the reference's OWN
utils.evaluate_error (/root/reference/cspn_pytorch/utils.py:19-47) and Wighted_L1_Loss (loss.py:16-23, forward and the
gradient autograd gives through it) on seeded inputs.  Build container only (needs /root/reference):

    python tests/golden/make_golden_metrics.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
REF = '/root/reference/cspn_pytorch'
HERE = os.path.dirname(os.path.abspath(__file__))
KEYS = ['MSE', 'RMSE', 'MAE', 'ABS_REL', 'DELTA1.02', 'DELTA1.05', 'DELTA1.10', 'DELTA1.25', 'DELTA1.25^2', 'DELTA1.25^3']


def main():
    from run_reference_eval import _stub_modules
    _stub_modules()                                  # utils.py imports matplotlib / skimage, absent here
    sys.path[:0] = [REF, os.path.join(REF, 'models')]
    import loss as ref_loss
    import utils as ref_utils
    cases = {
        'nyu_like': (3, (1, 1, 228, 304), 0.0, 1.0),          # dense ground truth
        'kitti_like': (4, (2, 1, 64, 256), 0.7, 1.0),         # 70 % of the ground truth missing (== 0)
        'close_prediction': (5, (1, 1, 40, 60), 0.2, 0.02),   # errors around the delta thresholds
        'nothing_valid': (6, (1, 1, 8, 8), 1.0, 1.0),
    }
    for name, (seed, shape, p_missing, noise) in cases.items():
        g = torch.Generator().manual_seed(seed)
        gt = torch.rand(shape, generator=g) * 10
        gt = gt * (torch.rand(shape, generator=g) >= p_missing).float()
        pred = (gt + noise * torch.randn(shape, generator=g)).clamp_min(0.05) if noise < 1 else torch.rand(shape, generator=g) * 10
        err = ref_utils.evaluate_error(gt_depth=gt, pred_depth=pred)
        vals = np.array([float(err[k]) for k in KEYS], dtype=np.float64)
        rec = dict(gt=gt.numpy(), pred=pred.numpy(), metrics=vals, keys=np.array(KEYS))
        if (gt > 0.0001).any():
            p = pred.clone().requires_grad_(True)
            loss = ref_loss.Wighted_L1_Loss()(p, gt)
            loss.backward()
            rec.update(loss=np.float64(loss.item()), grad_pred=p.grad.numpy())
        np.savez_compressed(os.path.join(HERE, 'metrics', name + '.npz'), **rec)
        print(name, dict(zip(KEYS, np.round(vals, 5))))


if __name__ == '__main__':
    main()
