"""Data-parallel training step on real GPUs: torchrun --nproc-per-node N tools/dp_train_check.py
Every rank trains on its shard of one global batch (fused forward / backward, NCCL all-reduce of the head gradients,
ClipAdam), eagerly and from a CUDA graph; the weights must stay identical across ranks and match a single-process run of
the whole batch on rank 0 (equal shard sizes: the mean of the shard means is the global mean).
--objective wsd: objective.WSD, whose voicing threshold comes from the loudest frame of the whole batch -- the all-reduce(max)
of that frame energy runs inside the step (and inside the captured graph) on every rank."""
import argparse, os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import speech_enhancement_by_s3prl_b200 as se
from speech_enhancement_by_s3prl_b200 import dp, synth

ap = argparse.ArgumentParser()
ap.add_argument("--objective", choices=["sisdr", "wsd"], default="sisdr")
args = ap.parse_args()
rank, world = dp.init_from_env()
dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
torch.cuda.set_device(dev)
pre = se.OnlinePreprocessor(sample_rate=16000, win_ms=32, hop_ms=16, n_freq=257).to(dev)
pre.channel_inp, pre.channel_tar = 0, 1
B = 8 * world
lengths, wavs = synth.batch(B, 2.0)
crit = se.WSD() if args.objective == "wsd" else se.SISDR()


def run(l, w, graph, steps=6):
    torch.manual_seed(1337)
    head = se.LinearResidual(input_size=257, output_size=257, precision=1).to(dev)
    eng = se.EnhancementEngine(pre, head, log_features=True, precision=1)
    opt = se.ClipAdam(head.parameters(), lr=1e-3)
    for _ in range(steps):
        loss = (eng.train_step_graph if graph else eng.train_step)(l, w, crit, opt, 1.0)
    torch.cuda.synchronize()
    return head.linear.weight.detach().clone(), loss.item()


l_s, w_s = dp.shard_batch(lengths, wavs, rank, world)
out = {}
for graph in (False, True):
    w_dp, loss = run(l_s.to(dev), w_s.to(dev), graph, steps=6 if not graph else 3)   # graph: 3 eager warm-ups + 3 replays
    gathered = [torch.empty_like(w_dp) for _ in range(world)]
    dist.all_gather(gathered, w_dp)
    spread = max((g - gathered[0]).abs().max().item() for g in gathered)
    out[graph] = (w_dp, spread, loss)
if rank == 0:
    saved = (dist.is_initialized(), )
    # single-process reference on the whole batch: switch the collectives off by running with world size 1 semantics
    import speech_enhancement_by_s3prl_b200.dp as dpm
    orig = dpm.allreduce_gradients, dpm.global_max
    dpm.allreduce_gradients, dpm.global_max = (lambda *a, **k: None), (lambda t: t)
    w_one, loss_one = run(lengths.to(dev), wavs.to(dev), False, steps=6)
    dpm.allreduce_gradients, dpm.global_max = orig
    for graph in (False, True):
        w_dp, spread, loss = out[graph]
        diff = (w_dp - w_one).abs().max().item()
        print(f"{args.objective} world {world} graph={graph}: max |w_rank - w_rank0| = {spread:.2e}, max |w_dp - w_single| = {diff:.2e}, "
              f"update size {(w_one - torch.nn.init.zeros_(w_one.clone())).abs().max().item():.2e}", flush=True)
        assert spread == 0.0, "ranks diverged"
        assert diff < 5e-4, "data-parallel training does not match the single-process step"
    print("dp_train_check OK", flush=True)
dist.barrier()
dist.destroy_process_group()
