"""torchrun check of the multi-GPU Kirchhoff on real GPUs: the sharded result (halo exchange: every rank receives only
its window of input columns; output blocks gathered to rank 0; exchanges overlapped with the kernels in bottom-up row
chunks) must equal, BIT FOR BIT, the unsharded image that rank 0 computes alone, for every pipeline depth, and so must
the round-1 scheme (full broadcast + all-gather).  Prints the timings of both schemes.  Finally repeats the bit-for-bit
checks with a layered velocity (synthetic.layered_velocity as per-sample RMS velocities).
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 scripts/check_sharded.py [S T]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from impdar_b200 import parallel, synthetic, migrationlib as ml

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank))))
S, T = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (4096, 16384)
tt, dk, _ = synthetic.geometry(S, T)
VEL = 1.69e8
if rank == 0:
    full = synthetic.diffractor_radargram(S, T, seed=9, n_diffractors=64)
    whole = ml.kirchhoff_device(full, tt, dk, VEL, False)          # the unsharded image
    kern = ml.kirchhoff_last_kernel()
else:
    full = whole = None

def x_for(exchange):
    if rank == 0:
        return full.clone()
    if exchange == "broadcast":
        return torch.zeros((S, T), dtype=torch.float32, device="cuda")
    return torch.empty((1, 1), dtype=torch.float32, device="cuda").expand(S, T)

PEER = {"halo": None, "halo-nopeer": False, "broadcast": None}      # peer_image argument: None = automatic, False = off

def run(exchange, chunks):
    x = x_for(exchange)
    out = parallel.kirchhoff_sharded_device(x, tt, dk, VEL, False, rank=rank, world=world, pipeline_chunks=chunks,
                                            exchange=exchange.split("-")[0], peer_image=PEER[exchange],
                                            gather=True if exchange == "broadcast" else 'src')
    torch.cuda.synchronize()
    return out

def timed(exchange, chunks, n=3):
    run(exchange, chunks); run(exchange, chunks); dist.barrier()
    ts = []
    for _ in range(n):
        x = x_for(exchange)
        torch.cuda.synchronize(); dist.barrier()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        parallel.kirchhoff_sharded_device(x, tt, dk, VEL, False, rank=rank, world=world, pipeline_chunks=chunks,
                                          exchange=exchange.split("-")[0], peer_image=PEER[exchange],
                                          gather=True if exchange == "broadcast" else 'src')
        b.record(); torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b)], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); ts.append(t.item())
    return min(ts)

if rank == 0:
    print("%d x %d on %d GPUs; single-GPU kernel: %s" % (S, T, world, kern), flush=True)
VARIANTS = [("halo", 1), ("halo", 4), ("halo", parallel.DEFAULT_CHUNKS), ("halo-nopeer", 1),
            ("halo-nopeer", parallel.DEFAULT_CHUNKS), ("broadcast", 1), ("broadcast", 4)]
for exchange, chunks in VARIANTS:
    if True:
        got = run(exchange, chunks)
        if exchange == "halo" and chunks == 1 and rank == 0:
            print("peer-mapped output image active: %s; ranges %s" % (parallel.peer_output_active(),
                  parallel.kirchhoff_output_ranges(T, world, tt, dk, VEL)), flush=True)
        if exchange == "halo":                           # the persistent image must not leak a previous call's rows
            got2 = run(exchange, chunks)
            if rank == 0 and not torch.equal(got, got2):
                print("SECOND CALL DIFFERS", flush=True)
        ok = torch.tensor([1.0 if (rank != 0 or torch.equal(got, whole)) else 0.0], device="cuda")
        if exchange == "broadcast" and rank != 0:       # every rank holds the image in the round-1 scheme
            ok[0] = 1.0 if got.shape == (S, T) else 0.0
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if rank == 0:
            print("exchange=%s pipeline_chunks=%s: sharded == unsharded bit for bit: %s" % (exchange, chunks, ok.item() == 1.0), flush=True)
for exchange, chunks in VARIANTS:
    if True:
        ms = timed(exchange, chunks)
        if rank == 0:
            print("exchange=%s pipeline_chunks=%s: %.2f ms" % (exchange, chunks, ms), flush=True)
# a different radargram through the same persistent image: a row copied before its owner has stored it would still
# hold the previous call's value (scaling by 2 is exact in float32, so the expected image is known bit for bit)
if rank == 0:
    full.mul_(2.0)
    whole.mul_(2.0)
for chunks in (1, parallel.DEFAULT_CHUNKS):
    got = run("halo", chunks)
    ok = torch.tensor([1.0 if (rank != 0 or torch.equal(got, whole)) else 0.0], device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("exchange=halo pipeline_chunks=%s, next radargram through the same image: bit for bit: %s" % (chunks, ok.item() == 1.0), flush=True)
# layered velocity: one RMS velocity per sample, passed through every layer (ranges, windows, kernels)
from impdar_b200 import RadarData
geo = RadarData(np.zeros((S, 1), np.float32), dt=synthetic.DT, travel_time=tt, dist=dk[:1])
VEL = ml.rms_velocity(tt, ml.getVelocityProfile(geo, synthetic.layered_velocity(tt)))
if rank == 0:
    whole = ml.kirchhoff_device(full, tt, dk, VEL, False)
    print("layered velocity %.3e .. %.3e; single-GPU kernel: %s" % (VEL.max(), VEL.min(), ml.kirchhoff_last_kernel()),
          flush=True)
for exchange, chunks in VARIANTS:
    got = run(exchange, chunks)
    ok = torch.tensor([1.0 if (rank != 0 or torch.equal(got, whole)) else 0.0], device="cuda")
    if exchange == "broadcast" and rank != 0:
        ok[0] = 1.0 if got.shape == (S, T) else 0.0
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("layered: exchange=%s pipeline_chunks=%s: sharded == unsharded bit for bit: %s" % (exchange, chunks, ok.item() == 1.0), flush=True)
parallel.free_exchange_buffers()
dist.destroy_process_group()
