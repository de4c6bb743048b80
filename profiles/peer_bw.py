"""Multi-GPU diagnostic (torchrun, one rank per GPU): where does the bandwidth of peer-memory row fetches go?

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 profiles/peer_bw.py

Brackets psb_peer_gather_rows (random rows of a row-sharded 16M x 128 table, 1M rows per rank) with what the same
box does for the same bytes: (a) cudaMemcpyAsync from the peer mapping (copy engine), (b) NCCL all_to_all_single,
(c) the gather kernel on SEQUENTIAL remote rows (pure P2P load stream), (d) on random rows, local rows only / remote
rows only / the mix."""
import ctypes
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, iters=5, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    t = torch.tensor([s.elapsed_time(e) / iters * 1e-3], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from prodsearch_b200 import _lib, peer
    from prodsearch_b200._lib import check, load, stream_ptr
    pg = peer.PeerGroup(device="cuda")
    rows, d, n = 16_000_000, 128, 1_000_000
    local_rows = (rows + world - 1) // world
    shard = pg.alloc(local_rows * d * 4)
    shard.view(torch.float32, (local_rows, d)).normal_()
    torch.cuda.synchronize()
    dist.barrier()
    out = torch.empty(n, d, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1 + rank)
    res = {"world": world}
    nxt = (rank + 1) % world

    def gather(ids):
        check(load().psb_peer_gather_rows(shard.ptr_array(), world, rows, d, ids.data_ptr(), ids.numel(), out.data_ptr(),
                                          None, -1, 0, None, stream_ptr()), "psb_peer_gather_rows")
    rb = n * d * 4
    cases = {
        "random_mixed": torch.randint(0, rows, (n,), device="cuda", generator=g),
        "random_remote_only": torch.randint(0, local_rows - 1, (n,), device="cuda", generator=g) * world + nxt,
        "random_local_only": torch.randint(0, local_rows - 1, (n,), device="cuda", generator=g) * world + rank,
        "sequential_remote": torch.arange(n, device="cuda") * world + nxt,
        "sequential_local": torch.arange(n, device="cuda") * world + rank,
    }
    for name, ids in cases.items():
        sec = timed(lambda: gather(ids))
        res["gather_" + name] = {"ms": round(sec * 1e3, 3), "GBps_rows_per_gpu": round(rb / sec / 1e9, 1)}
    # the bench's own construction: PeerShardedTable + host-generated uniform ids (profiles/r02l: 6.4 ms there)
    from prodsearch_b200 import synth
    from prodsearch_b200.peer import PeerShardedTable
    table = PeerShardedTable(rows + 1, d, pg, pad_idx=rows)
    with torch.no_grad():
        table.weight.normal_()
    table.weight.requires_grad_(False)
    idx = synth.gather_indices(n, rows, seed=11 + rank, dist="uniform").cuda()
    torch.cuda.synchronize()
    dist.barrier()

    def kernel_only(ids_, tab):
        check(load().psb_peer_gather_rows(tab.ptr_array(), world, rows + 1, d, ids_.data_ptr(), n, out.data_ptr(), None, -1, 0,
                                          None, stream_ptr()), "psb_peer_gather_rows")
    for name, ids_, tab in (("bench_table_bench_ids", idx, table.shard), ("bench_table_randint_ids", cases["random_mixed"], table.shard),
                            ("diag_shard_bench_ids", idx, shard)):
        sec = timed(lambda: kernel_only(ids_, tab))
        res["kernel_" + name] = {"ms": round(sec * 1e3, 3)}
    res["ids_stats"] = {"bench_unique": int(torch.unique(idx).numel()), "bench_max": int(idx.max()),
                        "randint_unique": int(torch.unique(cases["random_mixed"]).numel())}
    with torch.no_grad():
        sec = timed(lambda: table.fetch([idx]))
    res["fetch_bench_table"] = {"ms": round(sec * 1e3, 3)}
    # (a) copy engine from the peer mapping
    cudart = ctypes.CDLL("libcudart.so")
    src = shard.ptrs[nxt]
    sec = timed(lambda: cudart.cudaMemcpyAsync(ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(src), ctypes.c_size_t(rb),
                                               ctypes.c_int(3), ctypes.c_void_p(stream_ptr())))
    res["cudaMemcpyAsync_from_peer"] = {"ms": round(sec * 1e3, 3), "GBps": round(rb / sec / 1e9, 1)}
    # (b) NCCL all-to-all of the same bytes (n rows per rank, split evenly)
    a = torch.empty(n, d, device="cuda").normal_()
    b = torch.empty_like(a)
    sec = timed(lambda: dist.all_to_all_single(b, a))
    res["nccl_all_to_all_single"] = {"ms": round(sec * 1e3, 3), "GBps_per_gpu_total": round(rb / sec / 1e9, 1),
                                     "GBps_per_gpu_on_the_wire": round(rb * (world - 1) / world / sec / 1e9, 1)}
    if rank == 0:
        try:
            res["topo"] = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout.splitlines()[:4]
        except Exception as ex:                                                   # noqa: BLE001
            res["topo"] = str(ex)
        print(json.dumps(res), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
