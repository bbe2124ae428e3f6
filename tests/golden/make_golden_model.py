"""Model-level golden: the reference's OWN caller code -- resnet50 + Gudi UNet decoder of
/root/reference/cspn_pytorch/models/torch_resnet_cspn_nyu.py with the reference's own cspn.py as its last layer -- run here
on the CPU (seeded random weights, one random RGB-D input), recording exactly what the model hands to
post_process_layer (torch_resnet_cspn_nyu.py:372-375) and what the model returns.

    python tests/golden/make_golden_model.py      (build container only: needs /root/reference)

tests/golden/model/nyu_resnet50_tail.npz holds two 80x112 windows of the 228x304 image, at the top-left and the
bottom-right corner (so every image border is in one of them): guidance_<c> (1,8,80,112), blur_<c> and sparse_depth_<c>
(1,1,80,112), and out_<c>, the model's output on the part of the window at least `margin` = prop_time + 2 pixels from
its inner edges.  One step moves information by one pixel, so there the output depends on nothing outside the window.
tests/test_reference_model_golden_gpu.py feeds these boundary tensors to the B200 module and must reproduce the
reference MODEL's output -- the exit criterion of SURVEY.md section 7.2.
float16-rounded storage would break bit-faithfulness of the inputs, so everything is stored as float32 (npz-compressed).
"""
import importlib
import os
import sys

import numpy as np
import torch

REF_MODELS = '/root/reference/cspn_pytorch/models'
HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    assert os.path.isdir(REF_MODELS), 'reference tree not mounted'
    sys.path.append(REF_MODELS)                       # the reference's own cspn.py is what `import cspn` finds
    torch.Tensor.cuda = lambda self, *a, **k: self    # Unpool's ctor and cspn.py:50 call .cuda()
    torch.manual_seed(1234)
    model = importlib.import_module('torch_resnet_cspn_nyu')
    assert 'reference' in model.post_process.__file__
    net = model.resnet50(pretrained=False, cspn_config={'step': 24, 'norm_type': '8sum'}).eval()
    seen = {}
    layer = net.post_process_layer
    orig = layer.forward

    def spy(guidance, blur_depth, sparse_depth=None):
        seen.update(guidance=guidance.clone(), blur=blur_depth.clone(), sparse=sparse_depth.clone())
        return orig(guidance, blur_depth, sparse_depth)

    layer.forward = spy
    g = torch.Generator().manual_seed(99)
    x = torch.rand(1, 4, 228, 304, generator=g)
    x[:, 3] = x[:, 3] * 10 * (torch.rand(1, 228, 304, generator=g) < 500.0 / (228 * 304))   # nyu_dataset_loader.py:141-143
    with torch.no_grad():
        out = net(x)
    os.makedirs(os.path.join(HERE, 'model'), exist_ok=True)
    path = os.path.join(HERE, 'model', 'nyu_resnet50_tail.npz')
    np.savez_compressed(path, **windows(seen['guidance'], seen['blur'], seen['sparse'], out, 24), prop_time=24,
                        norm_type='8sum')
    print(path, os.path.getsize(path), 'bytes; out absmax', float(out.abs().max()), 'finite', bool(torch.isfinite(out).all()),
          'sparse points', int((seen['sparse'] > 0).sum()))


def windows(guidance, blur, sparse, out, prop_time, size=(80, 112)):
    H, W = out.shape[-2:]
    m = prop_time + 2
    rec = dict(image_hw=np.array([H, W]), margin=m)
    for c, r0, c0 in (('tl', 0, 0), ('br', H - size[0], W - size[1])):
        win = np.s_[..., r0:r0 + size[0], c0:c0 + size[1]]
        rec.update({f'guidance_{c}': guidance[win].numpy(), f'blur_{c}': blur[win].numpy(),
                    f'sparse_depth_{c}': sparse[win].numpy()})
        valid = np.s_[..., :size[0] - m, :size[1] - m] if c == 'tl' else np.s_[..., m:, m:]
        rec[f'out_{c}'] = np.ascontiguousarray(out[win].numpy()[valid])
    return rec


if __name__ == '__main__':
    main()
