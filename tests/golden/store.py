"""How the fixtures are stored and read back.

make_golden.py writes `compact(name, arrays)`: for the names in configs.STATE0_DIGEST_ONLY the reference's initial state_dict
(`state0.*`) becomes per-tensor SHA-1 digests (`state0sha.*`), and for the names in configs.SEEDED_WEIGHTS the coupling-network
weights and biases (`model.c<c>.k<k>.<net>.W<i>` / `.b<i>`) are left out.  `load(name)` puts those back: it builds this package's
BoostedFlow from the fixture's seed, accepts it only if its whole state_dict matches the reference's digests bit for bit, and takes
the weights from it.  Everything else in a fixture is the reference's own output, stored as made."""
import hashlib
import os
import re

import numpy as np

from .configs import CONFIGS, SEEDED_WEIGHTS, STATE0_DIGEST_ONLY, fixture_args

GOLDEN_DIR = os.path.dirname(os.path.abspath(__file__))
_NET_PARAM = re.compile(r"model\.c\d+\.k\d+\.\w+\.[Wb]\d+")


def _sha1(a):
    return np.frombuffer(hashlib.sha1(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def compact(name, arrays):
    """The stored form of a fixture's arrays (see the module docstring)."""
    out = {}
    for k, v in arrays.items():
        if k.startswith("state0.") and name in STATE0_DIGEST_ONLY:
            out["state0sha." + k[len("state0."):]] = _sha1(v)
        elif not (name in SEEDED_WEIGHTS and _NET_PARAM.fullmatch(k)):
            out[k] = v
    return out


def _seeded_net_params(name, g):
    import torch
    import gbnf_b200
    from oracle import gbnf_oracle as orc
    _, seed, _, toy_base = CONFIGS[name]
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        model = gbnf_b200.BoostedFlow(fixture_args(name))
    for k, v in model.state_dict().items():
        if not np.array_equal(_sha1(v.numpy()), g["state0sha." + k]):
            raise ValueError(f"{name}: the seeded constructor does not reproduce the reference's initial {k}")
    flat = orc.flatten_model(gbnf_b200.extract_model(model, toy_base=toy_base))
    return {"model." + k: v for k, v in flat.items() if _NET_PARAM.fullmatch("model." + k)}


def load(name):
    """The fixture `name` as {key: ndarray}, with every array the reference produced or started from."""
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))
    if name in SEEDED_WEIGHTS:
        g.update(_seeded_net_params(name, g))
    return g
