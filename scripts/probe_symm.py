#!/usr/bin/env python
"""2+ GPUs (torchrun): symmetric-memory gradient bucket + hand-written peer all-reduce vs NCCL — correctness and time."""
import ctypes, os, sys, traceback
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch
import torch.distributed as dist

rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
from easy_gaussian_splatting_b200 import _lib
lib = _lib.load()
n = 59 * 1_000_000
n_pad = (n + 4 * world - 1) // (4 * world) * (4 * world)
try:
    import torch.distributed._symmetric_memory as symm_mem
    group = dist.group.WORLD
    if hasattr(symm_mem, "enable_symm_mem_for_group"):
        try:
            symm_mem.enable_symm_mem_for_group(group.group_name)
        except Exception as e:
            print(rank, "enable_symm_mem_for_group:", repr(e)[:200])
    buf = symm_mem.empty(n_pad, dtype=torch.float32, device=dev)
    hdl = symm_mem.rendezvous(buf, group.group_name)
    print(rank, "rendezvous ok: world", hdl.world_size, "rank", hdl.rank, "ptrs", [hex(p) for p in hdl.buffer_ptrs],
          "multicast", getattr(hdl, "multicast_ptr", None), flush=True)
except Exception:
    traceback.print_exc()
    print(rank, "SYMM-MEM UNAVAILABLE", flush=True)
    dist.destroy_process_group()
    sys.exit(0)

g = torch.Generator(device=dev).manual_seed(100 + rank)
src = torch.randn(n_pad, device=dev, generator=g)
ref = src.clone()
dist.all_reduce(ref)
st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

def peer_allreduce():
    hdl.barrier(channel=0)
    rc = lib.egs_allreduce_f32_peer(world, rank, ctypes.c_void_p(hdl.buffer_ptrs_dev), n_pad, 0, st())
    assert rc == 0, lib.egs_last_error_string()
    hdl.barrier(channel=1)

buf.copy_(src)
peer_allreduce()
torch.cuda.synchronize()
err = (buf - ref).abs().max().item()
gathered = [torch.empty(8, device=dev) for _ in range(world)]
dist.all_gather(gathered, buf[:8].contiguous())
same = all(torch.equal(gathered[0], t) for t in gathered)
print(rank, f"max |peer - nccl| = {err:.3e}  (scale {ref.abs().max().item():.2f}); replicas identical: {same}", flush=True)

def tm(fn, reps=20):
    for _ in range(3): fn()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); e1.synchronize()
    return e0.elapsed_time(e1) / reps

def mm_allreduce():
    hdl.barrier(channel=0)
    rc = lib.egs_allreduce_f32_multimem(world, rank, ctypes.c_void_p(hdl.multicast_ptr), n_pad, 0, st())
    assert rc == 0, lib.egs_last_error_string()
    hdl.barrier(channel=1)

t_mm = None
if getattr(hdl, "multicast_ptr", 0):
    buf.copy_(src)
    mm_allreduce()
    torch.cuda.synchronize()
    err = (buf - ref).abs().max().item()
    dist.all_gather(gathered, buf[1000:1008].contiguous())
    print(rank, f"multimem: max |mm - nccl| = {err:.3e}; replicas identical: {all(torch.equal(gathered[0], t) for t in gathered)}", flush=True)
    t_mm = tm(mm_allreduce)
t_bar = tm(lambda: (hdl.barrier(channel=0), hdl.barrier(channel=1)))
t_peer = tm(peer_allreduce)
x = src.clone()
t_nccl = tm(lambda: dist.all_reduce(x))
if rank == 0:
    print(f"all-reduce of {n_pad * 4 / 1e6:.0f} MB on {world} GPUs: peer two-shot {t_peer:.3f} ms, multimem {t_mm} ms, NCCL {t_nccl:.3f} ms (two barriers alone {t_bar:.3f} ms)", flush=True)
dist.barrier()
dist.destroy_process_group()
