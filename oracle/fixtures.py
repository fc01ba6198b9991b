"""TEST INFRASTRUCTURE ONLY: readers for the compact fixtures (tests/golden/full_*.pt, reference_contract.json.gz) written
by oracle/gen_golden.py (which imports the real reference and therefore cannot be imported where the tests run)."""
import gzip
import json
import os
import zlib

import numpy as np
import torch


def load_full_labels(g):
    """-> list of [1,1,oh,ow] float label maps (the real reference's argmax masks, one per propagated frame)."""
    arr = np.frombuffer(zlib.decompress(g["ref_labels_zlib"]), dtype=np.uint8).reshape(g["ref_labels_shape"])
    return [torch.from_numpy(arr[i].copy()).float()[None, None] for i in range(arr.shape[0])]


def load_reference_contract(golden_dir):
    """-> {"models": {name: {"state_dict": {key: shape}, "config": {key: repr}}}, "palette": [...],
    "networks": {module path: [[imported module, [names]], ...]}} as recorded from the reference."""
    with gzip.open(os.path.join(golden_dir, "reference_contract.json.gz"), "rt") as fh:
        return json.load(fh)


def write_reference_standin(root, networks):
    """Write a stand-in for a reference checkout under `root`: every module of its ``networks`` package at its recorded path,
    holding the module's recorded ``from networks.* import`` statements and a placeholder for every name another module
    imports from it.  Enough to resolve imports through the package exactly as the reference's files do."""
    provided = {}
    for imports in networks.values():
        for mod, names in imports:
            provided.setdefault(mod, set()).update(names)
    for rel, imports in networks.items():
        mod = rel[:-len(".py")].replace("/", ".").removesuffix(".__init__")
        own = {n for _, names in imports for n in names}
        lines = [f"from {m} import {', '.join(names)}" for m, names in imports]
        lines += [f"{n} = None" for n in sorted(provided.get(mod, set()) - own)]
        path = os.path.join(root, rel)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as fh:
            fh.write("\n".join(lines) + "\n")
