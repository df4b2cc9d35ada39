"""CPU oracle of the field-transform hot path — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of
`bench.py` may import this package, and only as the checker or as the timed CPU baseline.
Nothing under `anemoi-transform_b200/` imports it; the product path has no CPU fallback.

Contents
    pointwise.py   numpy restatement of the earthkit-meteo formulas the pointwise filters call
    spmm.py        scipy call of the reference + sequential-accumulation restatement of csr_matvec
    spatial.py     restatement of reference spatial.py on scipy.spatial.cKDTree
    csr_matvec.c   plain-C restatement of scipy's csr_matvec / csr_matvecs (+ OpenMP driver)
    refstubs/      stub packages (earthkit.*, anemoi.utils) that let the UNMODIFIED reference
                   be imported from ANEMOI_REFERENCE_SRC (reference_import.py)
    make_golden.py runs the imported reference and writes tests/golden/*.npz

Pinning: see each module's header and DESIGN.md §7.
"""
