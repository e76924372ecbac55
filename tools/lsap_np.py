"""Plain restatement of scipy.optimize.linear_sum_assignment (scipy/optimize/rectangular_lsap: shortest augmenting
path, D. F. Crouse, "On implementing 2D rectangular assignment algorithms", IEEE TAES 2016).

The device solver of csrc/match.cu mirrors this loop step for step, so it documents the exact algorithm - order of the
double additions, the tie-break of the column choice, the swap-with-last removal from `remaining` - and a CPU test pins
it to scipy.  Slow (pure Python loops): meant for small matrices."""
import numpy as np


def linear_sum_assignment_np(cost):
    c = np.asarray(cost, dtype=np.float64)
    if c.ndim != 2:
        raise ValueError(f"expected a matrix (2-D array), got a {c.ndim} array")
    if c.size == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    transposed = c.shape[1] < c.shape[0]
    if transposed:
        c = c.T
    if np.any(np.isnan(c) | np.isneginf(c)):
        raise ValueError("matrix contains invalid numeric entries")
    nr, nc = c.shape
    u, v = np.zeros(nr), np.zeros(nc)
    col4row, row4col, path = np.full(nr, -1), np.full(nc, -1), np.full(nc, -1)
    for cur in range(nr):
        min_val, remaining, nrem = 0.0, list(range(nc - 1, -1, -1)), nc
        spc, sr, sc = np.full(nc, np.inf), np.zeros(nr, bool), np.zeros(nc, bool)
        i, sink = cur, -1
        while sink == -1:
            sr[i] = True
            lowest, index = np.inf, -1
            for it in range(nrem):
                j = remaining[it]
                r = min_val + c[i, j] - u[i] - v[j]   # ((minVal + c) - u) - v, left to right
                if r < spc[j]:
                    path[j], spc[j] = i, r
                if spc[j] < lowest or (spc[j] == lowest and row4col[j] == -1):
                    lowest, index = spc[j], it
            min_val = lowest
            if min_val == np.inf:
                raise ValueError("cost matrix is infeasible")
            j = remaining[index]
            if row4col[j] == -1:
                sink = j
            else:
                i = row4col[j]
            sc[j] = True
            nrem -= 1
            remaining[index] = remaining[nrem]
        u[cur] += min_val
        for k in np.flatnonzero(sr):
            if k != cur:
                u[k] += min_val - spc[col4row[k]]
        v[sc] -= min_val - spc[sc]
        j = sink
        while True:
            i = path[j]
            row4col[j] = i
            col4row[i], j = j, col4row[i]
            if i == cur:
                break
    if transposed:
        order = np.argsort(col4row)
        return col4row[order].astype(np.int64), order.astype(np.int64)
    return np.arange(nr, dtype=np.int64), col4row.astype(np.int64)
