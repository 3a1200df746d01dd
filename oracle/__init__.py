"""TEST INFRASTRUCTURE: CPU restatement of the reference (oracle.py / adcensus_oracle.c), the
shim that builds the reference itself (refshim/, Makefile, _ref/), its driver (refdriver.py) and
the stored outputs of its kernels (reference_outputs.py).
Only tests/, __graft_entry__.smoke() and bench.py's baseline legs may import this package."""
