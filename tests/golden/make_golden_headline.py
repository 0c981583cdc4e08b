"""Writes headline_port.npz: a fixed sample (util.headline_sample) of the outputs of the oracle port of upstream's forward
(net.EffiMVSPlus + OracleHotPath, fp32, TF32 off) at the two headline shapes, on the seed-11 samples tests/test_gpu_upstream.py
uses.  These are the port's outputs, not upstream's: upstream's source is not part of the repository.  Where it is not
staged, test_oracle_table_vs_upstream_full_shape compares the port with this sample, so that a change to the port at these
shapes shows; whether the port agrees with upstream there is checked only where upstream is staged.

    python tests/golden/make_golden_headline.py [out.npz]        # needs a CUDA device
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.dirname(os.path.dirname(HERE)), os.path.dirname(HERE)]

import effimvs_b200  # noqa: E402,F401
from effimvs_b200 import synthetic  # noqa: E402
from oracle import hotpath as ohp  # noqa: E402
from util import dtu_model, headline_sample  # noqa: E402


@torch.no_grad()
def main(out=os.path.join(HERE, "headline_port.npz")):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    arrays = {}
    for shape, ndepths in (("dtu", "48,8,8"), ("tanks", "96,8,8")):
        s = synthetic.make_sample(shape, seed=11, device="cuda")
        res = dtu_model(ohp.OracleHotPath(), "cuda", ndepths)(s["imgs"], s["proj_matrices"], s["depth_values"])
        for i, a in enumerate(headline_sample(res["depth"], res["photometric_confidence"])):
            arrays["{}_{:02d}".format(shape, i)] = a
    np.savez_compressed(out, **arrays)
    print("wrote", out, sum(a.nbytes for a in arrays.values()), "bytes")


if __name__ == "__main__":
    main(*sys.argv[1:2])
