"""CPU oracle for the dvd_b200 hot path — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference` leg may
import this package. The product path (dynamic-video-depth_b200/) never does.
Parity status: PINNED — every function here is checked against outputs of the reference's own
PyTorch code, stored as fixtures under tests/golden/ by oracle/gen_golden.py
(tests/test_oracle_vs_reference.py, tests/test_oracle_golden.py, tests/test_oracle_step.py).
"""
