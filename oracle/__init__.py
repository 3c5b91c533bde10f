"""CPU oracle for the message-passing hot path of kaddly/GraphNeuralNetwork.

TEST INFRASTRUCTURE ONLY.  Nothing under `oracle/` is imported by the product package
`graphneuralnetwork_b200`; only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` /
`--impl reference` legs of `bench.py` may import it, and only as the checker / the timed CPU
baseline.  The product path has no CPU fallback.

What it is: a restatement, on the CPU with numpy / scipy / torch-CPU, of the arithmetic the
reference layers perform (the reference's arithmetic *is* ATen + SciPy calls; the de-facto
pin is this image: torch 2.11.0, scipy 1.18.1, numpy 2.3.5 — SURVEY.md §8c).  Each function
cites the reference file:line it follows.

Pinning: the reference ships no tests, golden vectors or fixtures ("parity unpinned" by the
reference's own tests).  The oracle is therefore pinned against the reference ITSELF:
`oracle/ref_loader.py` imports the unmodified modules from a reference checkout named by
$GNN_REFERENCE_ROOT (the reference is not part of this repository) and
`tests/test_oracle_vs_reference_live.py` compares them with this restatement on seeded inputs;
`tests/golden/make_golden.py` dumps reference outputs into `tests/golden/*.npz`, which pin the
oracle wherever the reference is absent.
"""
