"""Generate tests/golden/reference_pcpr.npz by running THE REFERENCE'S OWN rasterizer kernel (pcpr.forward) on a B200.

    python tests/golden/make_reference_pcpr.py [OUT.npz]

It needs the reference extension that oracle/build_ref.py compiles into oracle/_ref/ where the reference sources are.

It records what tests/test_gpu_reference_kernel.py compares against: the reference kernel's index and depth maps of that
test's collision-free and dense scenes, with a checksum of each scene.  The dense scene has pixel contention, under which
the reference kernel is nondeterministic: the file holds one of its possible results.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import build_ref                                                    # noqa: E402
import test_gpu_reference_kernel as t                                           # noqa: E402


def main(out):
    pcpr = build_ref.load()
    if pcpr is None:
        raise SystemExit("oracle/_ref/pcpr*.so is not built (oracle/build_ref.py)")
    res = {}
    for name, (xyz, M), W, H in (("free", t.collision_free_scene(), t.FREE_W, t.FREE_H),
                                 ("dense", t.dense_scene(), t.DENSE_W, t.DENSE_H)):
        index, depth = pcpr.forward(torch.from_numpy(xyz), torch.from_numpy(M), W, H, 512)
        res.update({f"{name}_index": index.numpy(), f"{name}_depth": depth.numpy(),
                    f"{name}_checksum": np.array(t.checksum(xyz, M))})
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    np.savez_compressed(out, **res)
    print(out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_pcpr.npz"))
