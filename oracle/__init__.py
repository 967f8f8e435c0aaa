"""oracle/ — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A CPU restatement of the reference's scoring hot path (SURVEY.md §8), used ONLY as the checker:
`tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of `bench.py`
may import it.  Nothing under `deeprecommendation_b200/` imports `oracle` — the product path fails
loudly when the CUDA library is missing instead of falling back to anything here.

Contents
  restatement.py   torch-CPU / numpy restatement of the reference algorithm, function by function,
                   each citing the reference file:line it follows.  Travels to the GPU box.
  ref_loader.py    imports the UNMODIFIED reference modules from the src/ of a checkout of the original
                   project named by B200REC_REFERENCE_ROOT (not part of this repository) with `pyg_shim/`
                   standing in for the uninstallable torch_geometric 2.0.4.
  pyg_shim/        restatement of the five PyG symbols the reference touches.
  make_golden.py   runs the real reference (through ref_loader) on seeded synthetic inputs and writes
                   the fixtures under tests/golden/.  Committed together with the fixtures.
  synth.py         seeded synthetic generators for BASELINE.json's configs (SURVEY.md §8d).

Pinning status (SURVEY.md §8c): the reference ships NO tests, golden vectors or known-answer
fixtures for this path.  The restatement is therefore pinned against *outputs of the reference
itself executed in this container* (tests/golden/*.npz, produced by make_golden.py):
  - BasicNCF / AttentionNCF / MLP builder / dynamic collate / create_graph: the unmodified reference
    source runs under torch 2.11 + pandas 3.0 -> PINNED.
  - GraphNCF / LightGCNConv: the reference source runs unmodified, but its message passing executes
    inside torch_geometric 2.0.4 (env.yml:122), which is absent; pyg_shim/ restates it -> the
    GraphNCF arithmetic is "parity unpinned" at the PyG boundary (said again in DESIGN.md).
"""
