"""Generate tests/golden/reference_modules.npz by running THE REFERENCE'S OWN torch modules (READ/models).

    python tests/golden/make_reference_modules.py PATH_TO_REFERENCE_CHECKOUT

It records what tests/test_oracle_pin_reference.py compares against: the layout of the reference UNet's state_dict
(keys, shapes, dtypes), the reference UNet's output on the seeded inputs of the tests under the synthetic weights
(read_b200.synth, identified by their checksum), and one PointTexture lookup together with its random texture.
"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_modules.npz")


def main(ref_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, ref_dir)
    sys.modules.setdefault("imageio", types.ModuleType("imageio"))
    from READ.models.unet import UNet
    from READ.models.texture import PointTexture
    from read_b200 import synth

    torch.manual_seed(synth.SEED)
    sd = synth.synth_state_dict(synth.SEED)
    ref_sd = UNet().state_dict()
    keys = sorted(ref_sd)
    shapes = np.full((len(keys), 4), -1, np.int64)
    for i, k in enumerate(keys):
        shapes[i, :ref_sd[k].dim()] = ref_sd[k].shape
    dtypes = np.array([str(ref_sd[k].dtype).replace("torch.", "") for k in keys])

    net = UNet()
    net.load_state_dict(sd, strict=True)
    net.eval()
    g = torch.Generator().manual_seed(7)                                # test_unet_oracle_equals_reference_module
    xs = [torch.rand((2, 8, 32 >> l, 48 >> l), generator=g) for l in range(5)]
    with torch.no_grad():
        unet_out = net(*xs)
    g = torch.Generator().manual_seed(11)                               # test_training_forward_of_our_unet_equals_reference
    xs = [torch.rand((1, 8, 32 >> l, 32 >> l), generator=g) for l in range(4)]
    train_out = net(*xs).detach()

    g = torch.Generator().manual_seed(3)                                # test_gather_oracle_equals_reference_module
    tex = PointTexture(8, 500, init_method='rand')
    ids = torch.randint(0, 500, (3, 1, 9, 7), generator=g).float()
    with torch.no_grad():
        gather_out = tex(ids)

    np.savez_compressed(OUT, sd_keys=np.array(keys), sd_shapes=shapes, sd_dtypes=dtypes,
                        sd_checksum=synth.state_dict_checksum(sd), unet_out=unet_out.numpy(), train_out=train_out.numpy(),
                        texture=tex.texture_.detach().numpy(), ids=ids.numpy(), gather_out=gather_out.numpy())
    print(OUT, len(keys), "state_dict entries", os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
