"""Shared helpers of the tree-search tests (test_search_cpu.py, test_gpu_search.py): positions and their true boards."""
import numpy as np


def true_boards(export):
    """True boards i8[G,N,N] (0 BLACK, 1 WHITE, 2 EMPTY) from an export's region planes (every stone carries a label)."""
    reg = np.asarray(export["regions"])
    inner = reg[:, :, 1:-1, 1:-1]
    b = np.full(inner.shape[:1] + inner.shape[2:], 2, np.int8)
    b[inner[:, 1] != 0] = 1
    b[inner[:, 0] != 0] = 0
    return b


def random_boards(rng, G, N):
    """Random preset boards (any stone counts, connections included) and sides to move."""
    fill = rng.uniform(0.0, 0.9, size=(G, 1, 1))
    stones = rng.uniform(size=(G, N, N)) < fill
    colour = rng.integers(0, 2, size=(G, N, N))
    return np.where(stones, colour, 2).astype(np.int8), rng.integers(0, 2, size=G).astype(np.int8)


ENV_KINDS = (  # (variant, agent_mode, opponent_first)
    (0, 0, False), (0, 0, True), (1, 0, False), (1, 1, False), (1, 2, False))


def env_kwargs(variant, agent_mode, opponent_first):
    return dict(variant=variant, agent_mode=agent_mode, opponent_first=opponent_first)


def env_steps(N):
    """Env steps that leave games at every stage (with auto-reset): about a third of a board's plies."""
    return max(2, N * N // 3)
