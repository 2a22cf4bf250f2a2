"""FLOAT-FRAME ORACLE — test infrastructure only (see float_oracle.py)."""
