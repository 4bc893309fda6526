"""CPU oracles (test infrastructure only).  See the header of each module.

Nothing under ``gptest_b200/`` may import this package: the product path is CUDA-only and
fails loudly when its extension is missing.
"""

# The golden vectors under tests/golden/ were computed with OpenBLAS on this many threads.  OpenBLAS splits its sums
# by thread count, so the last bits of the N=1024 results depend on it: make_golden.py and the bit-exact tests of
# tests/test_oracle.py run with this count, so that hosts with more or fewer cores reproduce them bit for bit.
GOLDEN_BLAS_THREADS = 8
