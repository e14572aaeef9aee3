"""The distributed solve of csrc/solve_krylov.cu for systems with n_upper unknowns per voxel (the multiplet emissions:
unknown = voxel * n_upper + state), restated in numpy over torch.distributed (TEST INFRASTRUCTURE: a model of the
algorithm and of what the ranks exchange, used by the CPU suite under gloo; the product path is the CUDA one).

The same iteration as tests/krylov_model.py -- one all-gather of the right-hand side rows, one of the preconditioner's
block entries, one of the product's pieces per GMRES step, everything else redundant on every rank -- with the
preconditioner's blocks generalised to runs of radial voxels of one SZA column with all their states (pc_blocks).  With
n_upper = 1 and at most 128 radial voxels the blocks are krylov_model's SZA columns and the arithmetic is the same, bit
for bit (tests/test_multiplet_krylov_gloo.py checks it)."""
import numpy as np

from krylov_model import _assemble


def pc_blocks(n_r, n_col, n_upper=1, max_nr=128):
    """the unknowns of each diagonal block of the preconditioner, SZA column by column: every column cut, from the lowest
    voxel up, into runs of max_nr // n_upper radial voxels with all their states (the last run shorter).  Runs as equal
    as whole voxels allow took as many or more steps (H multiplet, 40x20 grid: 31 against 23)."""
    run_vox = min(n_r, max_nr // n_upper)
    out = []
    for j in range(n_col):
        for i0 in range(0, n_r, run_vox):
            vox = np.arange(i0, min(n_r, i0 + run_vox)) * n_col + j
            out.append((vox[:, None] * n_upper + np.arange(n_upper)[None, :]).ravel())
    return out


def solve(dist, world, rows, K_rows, branching, S0, n_r, n_col, tol=1e-13, max_it=160, precondition=True, n_upper=1):
    """rows: the voxels this rank built; K_rows = K[unknowns of those voxels, :] (n_upper rows per voxel, unknown = voxel *
    n_upper + state).  -> (S, steps, true relative residual)"""
    n = n_r * n_col * n_upper
    rows = (np.asarray(rows, dtype=np.int64)[:, None] * n_upper + np.arange(n_upper)[None, :]).ravel()
    A_rows = -branching * K_rows
    A_rows[np.arange(len(rows)), rows] += 1.0
    b = _assemble(dist, world, rows, S0[rows], n)
    Minv = None
    B_rows = A_rows
    if precondition:
        # block entries of the own rows: A[e][unknowns of the block of e]
        blocks = pc_blocks(n_r, n_col, n_upper)
        width = max(len(c) for c in blocks)
        block_of = np.empty(n, dtype=np.int64)
        for i, c in enumerate(blocks):
            block_of[c] = i
        entries = np.zeros((len(rows), width))
        for k, e in enumerate(rows):
            c = blocks[block_of[e]]
            entries[k, :len(c)] = A_rows[k, c]
        pre = _assemble(dist, world, rows, entries, n)                       # [n][width] on every rank
        Minv = [np.linalg.inv(pre[c][:, :len(c)]) for c in blocks]
        B_rows = np.array(A_rows)
        for c, Mi in zip(blocks, Minv):
            B_rows[:, c] = A_rows[:, c] @ Mi
    beta = np.sqrt(np.sum(b * b))
    if beta == 0:
        return np.zeros(n), 0, 0.0
    V = [b / beta]
    w_raw, inv_norm = b, 1.0 / beta
    g = np.zeros(max_it + 1); g[0] = beta
    cs, sn = np.zeros(max_it), np.zeros(max_it)
    R = np.zeros((max_it + 1, max_it))
    k = 0
    for j in range(max_it):
        x = w_raw * inv_norm
        w = _assemble(dist, world, rows, B_rows @ x, n)
        Vm = np.array(V)
        h1 = Vm @ w
        w = w - Vm.T @ h1
        w1sq = np.sum(w * w)
        h2 = Vm @ w
        w = w - Vm.T @ h2
        hn = np.sqrt(max(w1sq - np.sum(h2 * h2), 0.0))
        h = np.concatenate([h1 + h2, [0.0]])
        hi = h[0]
        for i in range(j):
            up = h[i + 1]
            h[i] = cs[i] * hi + sn[i] * up
            hi = -sn[i] * hi + cs[i] * up
        d = np.hypot(hi, hn)
        cs[j], sn[j] = (hi / d, hn / d) if d > 0 else (1.0, 0.0)
        h[j] = d
        R[:j + 1, j] = h[:j + 1]
        g[j + 1] = -sn[j] * g[j]
        g[j] = cs[j] * g[j]
        k = j + 1
        w_raw, inv_norm = w, (1.0 / hn if hn > 0 else 0.0)
        V.append(w * inv_norm)
        if abs(g[j + 1]) / beta <= tol or hn == 0:
            break
    y = np.linalg.solve(np.triu(R[:k, :k]), g[:k])
    u = np.array(V[:k]).T @ y
    S = u
    if precondition:
        S = np.zeros(n)
        for c, Mi in zip(blocks, Minv):
            S[c] = Mi @ u[c]
    AS = _assemble(dist, world, rows, A_rows @ S, n)
    return S, k, float(np.sqrt(np.sum((b - AS) ** 2)) / beta)
