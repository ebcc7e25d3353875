"""The reference arm: the UNMODIFIED google/TensorNetwork package, installed under oracle/_ref by
oracle/build_ref.py, plus the import environment it needs (baseline/refenv.py)."""
