"""Loads the fixtures of tests/golden/.  model_base.npz does not store its weights: they are the seeded initialisation of
make_golden.py's `_run_model`, regenerated here bit for bit and checked against the SHA-256 digest the fixture keeps of
the weights the reference ran with (tests/golden/make_golden.py, `shrink`)."""
import hashlib
import os

import numpy as np
import torch


class Fixture(dict):
    """The arrays of one .npz, with the `.files` list of numpy's NpzFile."""

    @property
    def files(self):
        return list(self)


def digest(arrays) -> str:
    h = hashlib.sha256()
    for k in sorted(arrays):
        a = np.asarray(arrays[k])
        h.update(f"{k} {a.dtype.str} {a.shape}\n".encode())
        h.update(a.tobytes(order="C"))
    return h.hexdigest()


def base_model_weights(H: int, W: int):
    """`sd.*` of model_base.npz: the reference's base_model initialisation under torch.manual_seed(0) (yogo_b200.YOGO
    draws from the generator in the same order), head weight x 0.05, BatchNorm affine U(.5, 1.5) / U(-.2, .2), conv
    biases U(-.1, .1), in that order."""
    import yogo_b200

    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        net = yogo_b200.YOGO((H, W), 0.0425, 0.0555, 7, clip_value=1.0)
        with torch.no_grad():
            net.model[-1].weight.mul_(0.05)
            for m in net.model.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.weight.uniform_(0.5, 1.5)
                    m.bias.uniform_(-0.2, 0.2)
                if isinstance(m, torch.nn.Conv2d) and m.bias is not None:
                    m.bias.uniform_(-0.1, 0.1)
    return {"sd." + k: v.numpy().copy() for k, v in net.state_dict().items()}


def load(golden_dir: str, name: str) -> Fixture:
    with np.load(os.path.join(golden_dir, name)) as npz:
        z = Fixture(npz.items())
    if "digest.sd" in z:
        sd = base_model_weights(*z["img"].shape[-2:])
        expect = str(z.pop("digest.sd"))
        assert digest(sd) == expect, (
            f"{name}: the regenerated weights are not the ones the reference ran with (torch's CPU generator or "
            "yogo_b200.YOGO's initialisation order changed)")
        z.update(sd)
    return z
