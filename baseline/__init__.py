"""The UNMODIFIED reference (vrettasm/VGPA), which is not part of this repository: a checkout named by
the environment variable VGPA_REFERENCE, or a copy in `baseline/_ref/` (git-ignored).  Nothing of the
product (`vgpa_b200/`) imports this package: it serves the drop-in tests (the reference's own objects
and optimiser driving the CUDA path), the golden-fixture scripts and `bench.py`'s reference figures."""
