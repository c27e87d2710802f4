"""CPU oracle for the rollout + PPO-update hot path of OpenRL.

TEST INFRASTRUCTURE ONLY.  A plain numpy / torch-CPU restatement of the reference's
algorithm, each function citing the reference file:line it follows.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s CPU-baseline legs may import it; the product
package `openrl_b200` never does (and fails loudly without its CUDA library).

Pinning: the reference ships no golden vectors for this path (SURVEY.md §0.5), so the oracle
is pinned against outputs of the unmodified reference executed in the build container
(`oracle/gen_golden.py` -> `tests/golden/*.npz`; checked by `tests/test_oracle_*.py`).
CartPole-v1 dynamics come from third-party gymnasium (absent): that one boundary is
"parity unpinned" (see oracle/cartpole_ref.py).
"""

# Intra-op thread count the traces under tests/golden were recorded with.  MKL partitions its GEMM reductions and the QR
# of `orthogonal_` by thread count, which moves last bits, so the bit-exact replays of those traces use the same count.
TRACE_THREADS = 8
