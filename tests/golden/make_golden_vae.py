"""Golden record of the reference `VAE` class's seeded initialisation and CPU forward, for
test_lib_cpu.py::test_vae_state_dict_layout, from the UNMODIFIED reference mpvae.py.

    python tests/golden/make_golden_vae.py [--reference DIR]   -> tests/golden/vae_init_forward.json

The reference is `DIR/mpvae.py`, by default the verbatim copy oracle/make_ref.py places under oracle/_ref/.  The
script fails when it is not there: the record must never come from mpvae_b200's own class.  The state_dict is recorded
as SHA-256 digests (it is 2.4 MB of weights), the forward's inputs and outputs as values; `source` names the file and
its SHA-256.
"""
import argparse
import hashlib
import importlib.util
import json
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
ARGS = dict(feature_dim=20, label_dim=7, latent_dim=5, z_dim=3, keep_prob=0.5, scale_coeff=1.0, residue_sigma="")


def digest(t):
    return hashlib.sha256(t.detach().contiguous().numpy().tobytes()).hexdigest()


def record(vae_class):
    """The seeded initialisation and forward of `vae_class` (the reference's VAE or a drop-in for it)."""
    np.random.seed(4)
    torch.manual_seed(0)
    vae = vae_class(SimpleNamespace(**ARGS))
    x = torch.randn(6, 20)
    y = (torch.rand(6, 7) < 0.3).float()
    torch.manual_seed(1)
    out = vae(y, x)
    return {
        "args": ARGS,
        "state_dict": [{"key": k, "dtype": str(t.dtype), "shape": list(t.shape), "sha256": digest(t)}
                       for k, t in vae.state_dict().items()],
        "x": x.tolist(), "y": y.tolist(),
        "forward": [o.detach().tolist() for o in out],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default=os.path.join(ROOT, "oracle", "_ref"),
                    help="directory holding the reference's unmodified mpvae.py")
    path = os.path.join(ap.parse_args().reference, "mpvae.py")
    if not os.path.exists(path):
        sys.exit(f"{path} not found: the record is made from the reference's mpvae.py only "
                 "(python oracle/make_ref.py --reference DIR installs the copy)")
    spec = importlib.util.spec_from_file_location("mpvae_reference_unmodified", path)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    rec = record(ref.VAE)
    with open(path, "rb") as f:
        rec["source"] = f"reference mpvae.py, sha256 {hashlib.sha256(f.read()).hexdigest()}"
    with open(os.path.join(HERE, "vae_init_forward.json"), "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
