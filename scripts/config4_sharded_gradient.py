"""BASELINE config 4's accurate path with the hypothesis set sharded over the ranks (torchrun): a 50 000-point grid,
top-k, `steps` steps of gradient ascent from each winner, arg-max.  Three methods, alternated in one run:
  sharded_gradient:  ShardedVerifier.refine_by_gradient with a PeerExchange (ahv_refine_gradient_sharded, one C call)
  sharded_perturb:   ShardedVerifier.refine (both passes sharded, m = 64 candidates per winner)
  one_gpu_gradient:  HypothesisVerifier.refine_by_gradient on this rank's GPU alone, over the whole set
for B in {1, 8, 32}, k in {4, 32}, min_sep_deg in {0, 30}.  Each time is the median of CUDA events over AHV_ITERS calls,
the largest over the ranks.  Every line records the card's name and power limit and whether the sharded gradient chain
equals the one-GPU result bit for bit on every rank.  One JSON line per configuration; rank 0 also writes them to
AHV_OUT when it is set.   AHV_N (50000), AHV_STEPS (20), AHV_ITERS (20)."""
import importlib, json, os, statistics, subprocess, sys, torch, torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
dev = torch.device("cuda", torch.cuda.current_device())
dist.init_process_group("nccl", device_id=dev)
ahv = importlib.import_module("3dahv_b200")
N, steps, iters = int(os.environ.get("AHV_N", "50000")), int(os.environ.get("AHV_STEPS", "20")), int(os.environ.get("AHV_ITERS", "20"))
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index)],
                     capture_output=True, text=True).stdout.strip()
grid = ahv.so3.grid_rotations(N, device=dev)
peer = ahv.dist.PeerExchange(32, dev, max_k=32, max_hyps=N)


def timed(fn):
    for _ in range(3):
        fn()
    dist.barrier(); torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    t = torch.tensor([statistics.median(a.elapsed_time(b) for a, b in ev)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def bits(ts):
    return [t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t for t in ts]


out_f = open(os.environ["AHV_OUT"], "w") if rank == 0 and os.environ.get("AHV_OUT") else None
for B in (1, 8, 32):
    W1, W2, b2, vs, _, _ = bench.synthetic_inputs(torch, B, 16)
    v = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    vs = vs.to(dev)
    vt = ahv.ops.rotate_volume(vs, ahv.so3.sample_rotations(B, seed=123, device=dev))   # config 4's known-rotation task
    one = ahv.HypothesisVerifier(W1.to(dev), W2.to(dev), b2.to(dev))
    sv = ahv.dist.ShardedVerifier(v, peer=peer)
    for k in (4, 32):
        for sep in (0.0, 30.0):
            def sharded():
                return sv.refine_by_gradient(vs, vt, grid, k=k, steps=steps, min_sep_deg=sep)

            def single():
                return one.refine_by_gradient(vs, vt, grid, k=k, steps=steps, min_sep_deg=sep)

            def perturb():
                return sv.refine(vs, vt, grid, k=k)

            ms = {"sharded_gradient": [], "sharded_perturb": [], "one_gpu_gradient": []}
            for _ in range(2):                                  # alternated twice
                ms["sharded_gradient"].append(timed(sharded))
                ms["sharded_perturb"].append(timed(perturb))
                ms["one_gpu_gradient"].append(timed(single))
            a, b = sharded(), single()
            ga = bits((a[0], a[1], a[2].topk_val, a[2].topk_idx, a[2].R_best, a[3], a[4]))
            gb = bits((b[0], b[1], b[2].topk_val, b[2].topk_idx, b[2].R_best, b[3], b[4]))
            eq = torch.tensor([int(all(torch.equal(x, y) for x, y in zip(ga, gb)))], device=dev)
            dist.all_reduce(eq, op=dist.ReduceOp.MIN)
            row = {"gpu": gpu, "world": world, "B": B, "N": N, "k": k, "min_sep_deg": sep, "steps": steps,
                   "ms": {m: min(t) for m, t in ms.items()}, "ms_runs": ms, "sharded_equals_one_gpu": bool(int(eq))}
            peer.check()                                        # raises if an exchange timed out
            if rank == 0:
                print(json.dumps(row), flush=True)
                if out_f:
                    out_f.write(json.dumps(row) + "\n")
if out_f:
    out_f.close()
dist.barrier()
peer.close()
dist.destroy_process_group()
