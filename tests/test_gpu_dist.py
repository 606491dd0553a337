"""2-GPU NCCL run of the sequence-parallel hot path (turbodiffusion_b200/dist.py): sharded block forward + K/V all-gather +
moment all-reduce must reproduce the single-GPU block output.  Skipped when fewer than 2 GPUs are visible."""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out_path, mode, dim, heads):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from turbodiffusion_b200.block import WanHotPath
    from turbodiffusion_b200.dist import SequenceParallel
    from turbodiffusion_b200.ops import wan_rope_angles
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ffn, thw = 512, (3, 10, 23)  # L = 690 -> 6 blocks of 128: ranks get 384 and 306 rows
    l = thw[0] * thw[1] * thw[2]
    g = torch.Generator().manual_seed(11)
    x = torch.randn(l, dim, generator=g).bfloat16().to(dev)
    e0 = (torch.randn(6, dim, generator=g) * 0.1).to(dev)
    ctx = torch.randn(64, dim, generator=g).bfloat16().to(dev)
    ang = wan_rope_angles(*thw, dim // heads, dev)
    model = WanHotPath(dim, ffn, heads, 2, dev, topk=0.4, seed=5)
    ref = model.step(x, e0, ang, ctx) if rank == 0 else None      # single-GPU result (no hook installed yet)
    sp = SequenceParallel(l, world, rank)
    assert sp.install(model, mode) == mode
    y_local = model.step(sp.scatter(x), e0, sp.scatter(ang), ctx)
    y = sp.gather_rows(y_local)
    torch.cuda.synchronize()
    if rank == 0:
        diff = (y.float() - ref.float())
        torch.save({"rel_l2": (diff.norm() / ref.float().norm()).item(), "max_abs": diff.abs().max().item(),
                    "rows": [sp.row_begin, sp.row_end]}, out_path)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode,dim,heads", [("allgather", 256, 2), ("ulysses", 256, 2), ("allgather", 384, 3),
                                            ("ulysses", 384, 3)])     # 3 heads over 2 ranks: the uneven head split
def test_sequence_parallel_matches_single_gpu(tmp_path, mode, dim, heads):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "sp.pt")
    mp.spawn(_worker, args=(2, port, out, mode, dim, heads), nprocs=2, join=True)
    res = torch.load(out)
    # identical arithmetic per row; only the fp32 summation order of the linear-attention moments differs (per-rank partial
    # sums, and the all-reduce in the all-gather mode), which moves the 16-bit kvw operand and through it many outputs by one unit in the
    # last place: measured 1e-3 .. 2.4e-3 (uneven-head split) with max |diff| = 1 bf16 ulp of the largest outputs
    assert res["rel_l2"] < 4e-3 and res["max_abs"] <= 0.0625, res
