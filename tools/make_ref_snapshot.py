#!/usr/bin/env python
"""Snapshot the reference files SURVEY.md §8(a) cites into the git-ignored `oracle/_ref/`.

The reference (kaddly/GraphNeuralNetwork) is Python and not part of this repository: nothing is compiled, the
files are copied verbatim from the checkout $GNN_REFERENCE_ROOT names (or the directory given on the command
line), so that a copy of the working tree carries them to a machine without that checkout.  `oracle/_ref/` is
test / baseline infrastructure (never imported by the product package): it lets
  * `bench.py --impl reference` time the reference's OWN collate_fn + GraphSage classes (kind "reference"),
  * `tests/test_reference_substitution_gpu.py` run the reference's own models and training loop with the
    drop-in layers substituted by import path, on the GPU.
Called by `__graft_entry__.build()`; a no-op when no reference checkout is named.  Never commits anything:
`oracle/_ref/` is listed in .gitignore.
"""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEST = os.path.join(ROOT, "oracle", "_ref")
# folder -> relative paths (files or directories of .py files) on or next to the hot path
FILES = {
    "GCN": ["GCN.py", "data_utils.py", "train_eval.py"],
    "GAT": ["models", "train_eval.py", "data_utils.py"],
    "GraphSAGE_Pytorch": ["models", "sample_utils.py", "data_utils.py", "train_eval.py"],
    "GraphSAGE": ["graph_utils.py", "GraphSAGE.py", "data_utils.py"],
    "HAN": ["models"],
    "GATNE_Pytorch": ["models/GATNE.py"],
    "GATNE": ["models/GATNE.py"],
    "GTN": ["models"],
}


def snapshot(src_root=None, dest=DEST) -> int:
    src_root = src_root or os.environ.get("GNN_REFERENCE_ROOT")
    if not src_root or not os.path.isdir(os.path.join(src_root, "GCN")):
        return 0
    n = 0
    for folder, rels in FILES.items():
        for rel in rels:
            src = os.path.join(src_root, folder, rel)
            dst = os.path.join(dest, folder, rel)
            if os.path.isdir(src):
                for name in sorted(os.listdir(src)):
                    if name.endswith(".py"):
                        os.makedirs(dst, exist_ok=True)
                        shutil.copyfile(os.path.join(src, name), os.path.join(dst, name))
                        n += 1
            elif os.path.isfile(src):
                os.makedirs(os.path.dirname(dst), exist_ok=True)
                shutil.copyfile(src, dst)
                n += 1
    with open(os.path.join(dest, "README.txt"), "w") as f:
        f.write("Verbatim copies of kaddly/GraphNeuralNetwork files made by tools/make_ref_snapshot.py.\n"
                "Git-ignored; test / baseline infrastructure only.\n")
    return n


if __name__ == "__main__":
    print(f"{snapshot(*(sys.argv[1:2]))} reference files -> {DEST}")
