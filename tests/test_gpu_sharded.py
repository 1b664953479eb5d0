"""One tensor spread over several ranks (SURVEY section 8e, row 2): the column-sharded sweep through
the C ABI (ndmps_ttsvd_sharded + ndmps_interleave_shards) against the single-GPU path.  world = 1
runs in-process; world = 2 spawns two ranks - NCCL when the box has two GPUs, otherwise both ranks
share the one GPU and the collectives go through gloo (same host logic, same kernels)."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from conftest import phantom                              # noqa: E402
from test_gpu_truncation import SHARDED_CUTOFF_CASE      # noqa: E402

ROOT = Path(__file__).resolve().parents[1]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _compare(sh, ref_obj, ref_rec, vol, factors, rank, world, tol):
    from imgcompressionmps.distributed import shard_volume
    assert sh.bond_sizes() == ref_obj.bond_sizes()
    for a, b in zip(sh.singular_values, ref_obj.singular_values):
        assert np.allclose(a, b, rtol=0, atol=tol * b[0])
    mine = sh.to_local_tensor_device()
    want = shard_volume(ref_rec, factors, rank, world)
    rel = float(torch.linalg.vector_norm((mine - want).double()) / torch.linalg.vector_norm(want.double()))
    assert rel < tol, rel
    return rel


@pytest.mark.parametrize("shape,chi,cutoff", [
    pytest.param((64, 64, 64), 16, 1e-10, id="shape0-16"),
    pytest.param((32, 48, 40), 12, 1e-10, id="shape1-12"),
    # an rsum2 cutoff that binds below chi (test_gpu_truncation.py::test_sharded_cutoff_case_is_decidable checks
    # that no threshold sits within rounding of a compared value)
    pytest.param(*SHARDED_CUTOFF_CASE, id="shape0-16-cutoff4e-3"),
])
def test_sharded_world1_equals_plain_sweep(shape, chi, cutoff):
    from imgcompressionmps.core.ndmps import NDMPS
    from imgcompressionmps.distributed import ShardedNDMPS
    from imgcompressionmps.utils.core import get_factorlist
    x = torch.from_numpy(phantom(shape, seed=3, background=0.01).astype(np.float32)).cuda()
    ref = NDMPS.from_tensor(x, max_bond=chi, cutoff=cutoff)
    sh = ShardedNDMPS.from_local(x, shape, rank=0, world=1, max_bond=chi, cutoff=cutoff, stop_bytes=1 << 16)
    factors, _ = get_factorlist(shape)
    _compare(sh, ref, ref.to_tensor_device(), x, factors, 0, 1, 1e-6)
    for a, b in zip(sh.cores, ref.mps.cores):
        assert a.shape == b.shape


def _worker(rank, world, port, shape, chi, out_dir):
    for p in (str(ROOT), str(ROOT / "img-compression-mps_b200"), str(ROOT / "tests")):
        sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    from conftest import phantom as ph
    from imgcompressionmps.core.ndmps import NDMPS
    from imgcompressionmps.distributed import ShardedNDMPS, shard_volume
    from imgcompressionmps.utils.core import get_factorlist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    two = torch.cuda.device_count() >= world
    torch.cuda.set_device(rank if two else 0)
    dist.init_process_group("nccl" if two else "gloo", rank=rank, world_size=world)
    x = torch.from_numpy(ph(shape, seed=9, background=0.01).astype(np.float32)).cuda()
    factors, _ = get_factorlist(shape)
    local = shard_volume(x, factors, rank, world).contiguous()
    sh = ShardedNDMPS.from_local(local, shape, max_bond=chi, stop_bytes=1 << 16)
    ref = NDMPS.from_tensor(x, max_bond=chi)                          # the whole tensor on this rank
    rel = _compare(sh, ref, ref.to_tensor_device(), x, factors, rank, world, 2e-6)
    np.save(Path(out_dir) / f"rank{rank}.npy", np.array(sh.bond_sizes() + [int(rel < 2e-6)]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("shape,chi", [((64, 64, 64), 16), ((128, 128, 128), 64)])
def test_sharded_two_ranks_match_single_gpu(tmp_path, shape, chi):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), shape, chi, str(tmp_path)), nprocs=2, join=True)
    a, b = np.load(tmp_path / "rank0.npy"), np.load(tmp_path / "rank1.npy")
    assert np.array_equal(a, b) and a[-1] == 1
