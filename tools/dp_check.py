"""Multi-GPU check, run under torchrun on N GPUs:  torchrun --nproc-per-node N tools/dp_check.py OUT.json
  1. NCCL all-reduce through the C-ABI communicator,
  2. replicated data on every rank  ==> the DP step equals the single-GPU step (gradient mean over ranks = the gradient),
  3. different data per rank        ==> all ranks hold bit-identical parameters after every step,
  4. the reference's parameter averaging (params + updater state) through b2g_net_average_parameters,
  5. sync_bn: W ranks x N/W images with pooled BatchNorm statistics == 1 GPU x N images (SURVEY.md 8e),
  6. the bf16 gradient payload and the overlapped two-bucket all-reduce (B2G_AR_OVERLAP=1 in the environment) keep ranks identical.
Rank 0 writes the results to OUT.json.  tests/test_gpu_dp.py runs it under torchrun when the machine has >= 2 GPUs."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist

import gan_deeplearning4j_b200 as b
from gan_deeplearning4j_b200 import models as m, parallel

OUT = sys.argv[1]
rank, world, local = parallel.env_rank_world()
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ctx = b.Context(local)
parallel.attach_communicator(ctx, dist, rank, world)
out = {"world": world}
a = ctx.allreduce_test(np.full(1000, rank + 1.0, np.float32))
assert np.allclose(a, world * (world + 1) / 2), a[:3]
out["allreduce"] = "ok"


def make(seed_shift, prec):
    n, size, z, nf = 16, 32, 16, 64
    gs, ds = m.dcgan_generator(size, z, nf, 3, lr=1e-3), m.dcgan_discriminator(size, nf, 3, lr=1e-3)
    G = b.Net(ctx, gs, (z,), max_batch=n, precision=prec, xent_clip_eps=0.0, seed=1)
    D = b.Net(ctx, ds, (3, size, size), max_batch=2 * n, precision=prec, xent_clip_eps=0.0, bn_groups=2, seed=2)
    if os.environ.get("B2G_P2P_AR", "1") != "0":        # collective: gradient all-reduce as one peer-memory kernel (CUDA IPC), else ncclAllReduce
        ok = [D.enable_p2p_allreduce(), G.enable_p2p_allreduce()]
        out["allreduce_transport"] = "peer-memory kernel" if all(ok) else "nccl (peer mapping unavailable)"
    else:
        out["allreduce_transport"] = "nccl"
    rng = np.random.default_rng(100 + seed_shift)
    data = [rng.uniform(-1, 1, (n, 3, size, size)), rng.uniform(-1, 1, (n, z)), rng.uniform(-1, 1, (n, z)),
            1 + 0.05 * rng.standard_normal((n, 1)), 0.05 * rng.standard_normal((n, 1)), np.ones((n, 1))]
    return G, D, b.Gan(G, D, use_cuda_graph=False), data


for prec, name in ((b.FP32, "fp32"), (b.BF16, "bf16")):
    # (2) replicated data
    G, D, gan, data = make(0, prec)
    for _ in range(3):
        l_dp = gan.step(*data)
    pG, pD = G.params(), D.params()
    gan.close(); G.close(); D.close()
    ref_ctx = b.Context(local)            # no communicator: the single-GPU step
    saved = ctx
    Gs = b.Net(ref_ctx, m.dcgan_generator(32, 16, 64, 3, lr=1e-3), (16,), max_batch=16, precision=prec, xent_clip_eps=0.0, seed=1)
    Ds = b.Net(ref_ctx, m.dcgan_discriminator(32, 64, 3, lr=1e-3), (3, 32, 32), max_batch=32, precision=prec, xent_clip_eps=0.0, bn_groups=2, seed=2)
    gs_ = b.Gan(Gs, Ds, use_cuda_graph=False)
    for _ in range(3):
        l_1 = gs_.step(*data)
    tol = 2e-3 if prec == b.FP32 else 5e-2
    dG = np.abs(pG - Gs.params()).max(); dD = np.abs(pD - Ds.params()).max()
    out[f"replicated_{name}"] = {"max_abs_dG": float(dG), "max_abs_dD": float(dD), "loss_dp": l_dp.tolist(), "loss_1gpu": l_1.tolist()}
    assert np.allclose(l_dp, l_1, atol=tol), (l_dp, l_1)
    assert dG < 3.1e-3 and dD < 3.1e-3, (dG, dD)      # Adam steps are ~lr=1e-3 each: sign-level agreement after 3 steps
    gs_.close(); Gs.close(); Ds.close(); ref_ctx.close()
    # (3) different data per rank: parameters stay bit-identical across ranks
    G, D, gan, data = make(1 + rank, prec)
    for _ in range(3):
        gan.step(*data)
    for net, tag in ((G, "G"), (D, "D")):
        p = torch.from_numpy(net.params()).cuda()
        lo, hi = p.clone(), p.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        out[f"sharded_{name}_{tag}_identical"] = bool(torch.equal(lo, hi))
        assert torch.equal(lo, hi), tag
    gan.close(); G.close(); D.close()
# (4) the reference's own rule: local fits, then parameters AND updater state averaged over ranks (J:325-330)
dspec = m.dcgan_discriminator(32, 64, 3, lr=1e-3)
net = b.Net(ctx, dspec, (3, 32, 32), max_batch=16, precision=b.FP32, xent_clip_eps=0.0, seed=2)
net.set_grad_allreduce(False)
rng = np.random.default_rng(500 + rank)
net.fit(rng.uniform(-1, 1, (16, 3, 32, 32)), rng.uniform(0, 1, (16, 1)))
before = torch.from_numpy(np.concatenate([net.params(), net.updater_state()])).cuda()
mean = before.clone(); dist.all_reduce(mean, op=dist.ReduceOp.SUM); mean /= world
net.average_parameters()
after = np.concatenate([net.params(), net.updater_state()])
err = float(np.abs(after - mean.cpu().numpy()).max())
out["parameter_averaging_max_abs_err"] = err
assert err < 1e-6, err
net.close()
# (5) sync_bn: the global batch of W*n images, rank r holding slice r, must train like one GPU holding all of it (BF16: the fused BatchNorm path)
n, size, z, nf = 16, 32, 16, 64
gs, ds = m.dcgan_generator(size, z, nf, 3, lr=1e-3), m.dcgan_discriminator(size, nf, 3, lr=1e-3)
rng = np.random.default_rng(900)
NG = n * world
full = [rng.uniform(-1, 1, (NG, 3, size, size)), rng.uniform(-1, 1, (NG, z)), rng.uniform(-1, 1, (NG, z)), 1 + 0.05 * rng.standard_normal((NG, 1)), 0.05 * rng.standard_normal((NG, 1)), np.ones((NG, 1))]
mine = [a[rank * n:(rank + 1) * n] for a in full]
G = b.Net(ctx, gs, (z,), max_batch=n, precision=b.BF16, xent_clip_eps=0.0, seed=1); D = b.Net(ctx, ds, (3, size, size), max_batch=2 * n, precision=b.BF16, xent_clip_eps=0.0, bn_groups=2, seed=2)
G.set_sync_bn(True); D.set_sync_bn(True)
gan = b.Gan(G, D, use_cuda_graph=False)
for _ in range(2):
    l_sync = gan.step(*mine)
pG, pD = G.params(), D.params()
gan.close(); G.close(); D.close()
one = b.Context(local)
G1 = b.Net(one, gs, (z,), max_batch=NG, precision=b.BF16, xent_clip_eps=0.0, seed=1); D1 = b.Net(one, ds, (3, size, size), max_batch=2 * NG, precision=b.BF16, xent_clip_eps=0.0, bn_groups=2, seed=2)
g1 = b.Gan(G1, D1, use_cuda_graph=False)
for _ in range(2):
    l_one = g1.step(*full)
dG = float(np.abs(pG - G1.params()).max()); dD = float(np.abs(pD - D1.params()).max())
mG = float(np.abs(pG - G1.params()).mean()); mD = float(np.abs(pD - D1.params()).mean())
lg = torch.tensor(np.asarray(l_sync, np.float64)).cuda(); dist.all_reduce(lg, op=dist.ReduceOp.SUM); lg = (lg / world).cpu().numpy()
out["sync_bn"] = {"max_abs_dG": dG, "max_abs_dD": dD, "mean_abs_dG": mG, "mean_abs_dD": mD, "loss_mean_over_ranks": lg.tolist(), "loss_1gpu_full_batch": np.asarray(l_one).tolist()}
# two Adam steps of lr 1e-3 (early Adam moves every weight by ~lr*sign(g)): an element whose gradient is numerically zero may flip sign in both
# steps (2 x 2*lr); everything else agrees to round-off, so the MEAN difference is orders of magnitude below one step
assert dG < 4.5e-3 and dD < 4.5e-3 and mG < 5e-5 and mD < 5e-5, (dG, dD, mG, mD)
assert np.allclose(lg, l_one, atol=3e-2), (lg, l_one)
g1.close(); G1.close(); D1.close(); one.close()
# (6) bf16 gradient payload: ranks stay identical, result close to the fp32 payload
G, D, gan, data = make(1 + rank, b.BF16)
G.set_grad_payload_bf16(True); D.set_grad_payload_bf16(True)
for _ in range(3):
    gan.step(*data)
for net, tag in ((G, "G"), (D, "D")):
    p = torch.from_numpy(net.params()).cuda(); lo, hi = p.clone(), p.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    out[f"bf16_payload_{tag}_identical"] = bool(torch.equal(lo, hi)); assert torch.equal(lo, hi), tag
gan.close(); G.close(); D.close()
out["ar_overlap_env"] = os.environ.get("B2G_AR_OVERLAP", "0")
if rank == 0:
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("dp_check ok", json.dumps(out)[:600])
ctx.close()
dist.destroy_process_group()
