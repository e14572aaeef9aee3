"""The distributed solve of the multiplet emissions on CPU: world size 2 and 3 over gloo (tests/krylov_multiplet_model.py:
n_upper states per voxel), with the oracle's multiplet K for O I 102.6 nm, the H Lyman multiplet and the singlet through
the multiplet code.  Each rank holds only the element rows of its interleaved shard of voxels; the result must be the
dense solution, the same on every rank.  The CUDA form is tested by tests/test_multiplet_distributed.py on the GPU box."""
import importlib
import os
import socket
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = "3d_planetary_rt_model_b200"
KINDS = [0, 1, 2]          # O_1026_emission, H_lyman_multiplet, H_lyman_singlet


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir, kind, drop_rows):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, HERE)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    synth = importlib.import_module(PKG + ".synth")
    multi = importlib.import_module(PKG + ".multi")
    import krylov_multiplet_model
    from oracle import multbind
    scn = synth.make_multiplet_scenario(kind, 20, 12, 6, 8, sza_T_contrast=0.1)
    O = multbind.OracleMultiplet(scn, "f64")
    O.build_rows()
    K, S0, nu = O.K(), O.vectors()["S0"], O.n_upper
    n_r, n_col = scn.n_rb - 1, scn.n_sb - 1
    rows = [v for a, b in multi.partition_interleaved(O.n_vox, world, rank, 3) for v in range(a, b)]
    if drop_rows and rank == world - 1:
        rows = rows[:-2]
    el = [v * nu + s for v in rows for s in range(nu)]
    res = {}
    try:
        for pc in (False, True):
            # the multiplet's branching is folded into K (multiplet_CFR_emission::pre_solve is empty): A = I - K
            res[pc] = krylov_multiplet_model.solve(dist, world, rows, K[el], 1.0, S0, n_r, n_col, precondition=pc, n_upper=nu)
        exact = np.linalg.solve(np.eye(O.n_el) - K, S0)
        for pc in (False, True):
            assert np.max(np.abs(res[pc][0] - exact)) <= 1e-10 * np.max(np.abs(exact)), pc
            assert res[pc][2] < 1e-12
        np.save(os.path.join(out_dir, f"S{rank}.npy"), np.stack([res[False][0], res[True][0]]))
        np.save(os.path.join(out_dir, f"steps{rank}.npy"), np.array([res[False][1], res[True][1]]))
    except RuntimeError as ex:
        with open(os.path.join(out_dir, f"error{rank}"), "w") as f:
            f.write(str(ex))
    dist.destroy_process_group()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("world", [2, 3])
def test_ranks_with_their_own_element_rows_reach_the_dense_solution(tmp_path, world, kind):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), kind, False), nprocs=world, join=True)
    S = [np.load(tmp_path / f"S{r}.npy") for r in range(world)]
    steps = [np.load(tmp_path / f"steps{r}.npy") for r in range(world)]
    assert steps[0][1] <= steps[0][0]                       # the block preconditioner takes no more steps than none
    for r in range(1, world):
        assert np.array_equal(S[0], S[r])                  # the ranks ran the same arithmetic on the same exchanged pieces
        assert np.array_equal(steps[0], steps[r])


def test_missing_element_rows_are_caught_by_the_census(tmp_path):
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), 1, True), nprocs=2, join=True)
    for r in range(2):
        assert "do not add up" in open(tmp_path / f"error{r}").read()


@pytest.mark.parametrize("n_r, n_upper, runs", [(99, 1, 1), (99, 3, 3), (99, 4, 4), (19, 4, 1), (200, 1, 2)])
def test_preconditioner_blocks_are_runs_of_whole_voxels(n_r, n_upper, runs):
    """every SZA column is cut into runs of 128 // n_upper radial voxels with all their states; the blocks partition the
    unknowns"""
    sys.path.insert(0, HERE)
    import krylov_multiplet_model
    n_col = 5
    blocks = krylov_multiplet_model.pc_blocks(n_r, n_col, n_upper)
    assert len(blocks) == n_col * runs
    assert max(len(c) for c in blocks) <= 128
    allc = np.concatenate(blocks)
    assert np.array_equal(np.sort(allc), np.arange(n_r * n_col * n_upper))
    for c in blocks:
        vox = c // n_upper
        assert len(set(vox % n_col)) == 1                     # one SZA column
        assert len(c) == n_upper * len(set(vox))              # whole voxels


def _singlet_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, HERE)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    synth = importlib.import_module(PKG + ".synth")
    multi = importlib.import_module(PKG + ".multi")
    import krylov_model
    import krylov_multiplet_model
    import oraclebind
    scn = synth.make_scenario(12, 8, 5, 6, n_em=1, sza_T_contrast=0.1)
    O = oraclebind.OracleModel(scn, "f64")
    O.build_rows()
    K, S0, w = O.K(0), O.vectors(0)["S0"], float(scn.em_scalars[0][0])
    n_r, n_col = scn.n_rb - 1, scn.n_sb - 1
    rows = [v for a, b in multi.partition_interleaved(scn.n_vox, world, rank, 3) for v in range(a, b)]
    same = []
    for pc in (False, True):
        a = krylov_model.solve(dist, world, rows, K[rows], w, S0, n_r, n_col, precondition=pc)
        b = krylov_multiplet_model.solve(dist, world, rows, K[rows], w, S0, n_r, n_col, precondition=pc)
        same.append(np.array_equal(a[0], b[0]) and a[1] == b[1] and a[2] == b[2])
    np.save(os.path.join(out_dir, f"same{rank}.npy"), np.array(same))
    dist.destroy_process_group()


def test_one_state_is_the_singlet_model_bit_for_bit(tmp_path):
    """n_upper = 1 on a grid of <= 128 radial voxels: the blocks are the SZA columns, the arithmetic that of
    krylov_model (the singlet model the CUDA singlet path is checked against)"""
    mp.spawn(_singlet_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        assert np.load(tmp_path / f"same{r}.npy").all()
