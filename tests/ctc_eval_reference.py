"""Reference dynamic programs for the ASR evaluation tests: the Levenshtein distance as a plain Python DP and as the
same recurrence vectorised over a row with numpy (exact: integer arithmetic), used where the plain DP is too slow."""
import numpy as np


def edit_distance_py(a, b):
    """Unit-cost Levenshtein distance, the textbook O(len(a) len(b)) table, one row at a time."""
    prev = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        cur = [i] + [0] * len(b)
        for j in range(1, len(b) + 1):
            cur[j] = min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (a[i - 1] != b[j - 1]))
        prev = cur
    return prev[-1]


def edit_distance_np(a, b):
    """The same table, row by row: with t[j] = min(D[i-1][j] + 1, D[i-1][j-1] + cost), the left-to-right term
    D[i][j] = min_k<=j (t[k] + j - k) is a running minimum of t[k] - k."""
    a, b = np.asarray(a, dtype=np.int64), np.asarray(b, dtype=np.int64)
    m = len(b)
    j = np.arange(m + 1, dtype=np.int64)
    prev = j.copy()
    for i in range(1, len(a) + 1):
        t = np.empty(m + 1, dtype=np.int64)
        t[0] = i
        t[1:] = np.minimum(prev[1:] + 1, prev[:-1] + (b != a[i - 1]))
        prev = np.minimum.accumulate(t - j) + j
    return int(prev[-1])
