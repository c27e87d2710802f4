"""Host-side index math of the joint-action (JRPO) update: `chunk_row_indices_v3` names the buffer rows that
recurrent_generator_v3 (replay_data.py:425-551) puts in a minibatch, in its (chunk, step, agent) order."""
import numpy as np
import torch

from openrl_b200.buffers.replay_data import chunk_row_indices_v3


def test_chunk_row_indices_v3_follow_cast_v3():
    T, N, A, L = 7, 3, 3, 4
    # buffer row t*N*A + n*A + a as a (T, N, A, 1) array, flattened the way _cast_v3 / _flatten_v3 do
    rows = np.arange(T * N * A).reshape(T, N, A, 1)
    cast = rows.transpose(1, 0, 2, 3).reshape(-1, A, 1)   # (N*T, A, 1): g = n*T + t
    ids = torch.tensor([4, 0, 2])
    want = np.stack([cast[c * L:c * L + L] for c in ids.numpy()], axis=1).reshape(-1)   # (L, n, A) -> rows (l*n + j)*A + a
    got = chunk_row_indices_v3(ids, L, T, N, A).numpy()
    # the kernels and the moments only need the same SET of rows per chunk step; the order here is (chunk, step, agent)
    assert sorted(got.tolist()) == sorted(want.tolist())
    by_chunk = got.reshape(len(ids), L, A)
    for j, c in enumerate(ids.tolist()):
        for l in range(L):
            g = c * L + l
            assert by_chunk[j, l].tolist() == [(g % T) * N * A + (g // T) * A + a for a in range(A)]
    agent0 = chunk_row_indices_v3(ids, L, T, N, A, agent0_only=True).numpy()
    assert agent0.tolist() == by_chunk[:, :, 0].reshape(-1).tolist()
