"""CPU oracle for the BP hot path -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this package.  The product (ldpcdecoders.jl_b200) never does.
PARITY UNPINNED: see the header of bp_oracle.c.
"""
from .oracle import (build, load, batch_decode, bposd_decode, bposd_order_decode, osd0_given, bpots_decode, sample, threshold, num_threads,  # noqa: F401
                     csc_arrays)
