"""Data-parallel equivalence (SURVEY.md §8e): the same global batch on 1 GPU and sharded by dialog over 2 GPUs
(one process per GPU, one NCCL all-reduce of the flat gradient inside vd_clamp_adam_step) must give the same
gradient and the same weights after the optimiser step, to fp32 reduction-order tolerance."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from helpers import small_batch, small_params

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


BIG = dict(rnnHiddenSize=256, embedSize=64, vocabSize=300, numOptions=100, commonEmbeddingSize=64, imgFeatureSize=64,
           imgSpatialSize=4, imgEmbedSize=32)          # option LSTM: 2 dialogs x 10 x 100 = 2000 rows per rank -> tensor-core kernels


def _case(enc, dec, mode, gpuid):
    p = small_params(enc, dec, gpuid=gpuid, **(BIG if mode != 1 else {}))
    return p, small_batch(p, B=4, seed=3)


def _worker(rank, world, port, enc, dec, mode, out):
    import torch.distributed as dist
    from visdial_b200 import Batch, Engine, init_parameters
    from visdial_b200 import dist as vdist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    p, full = _case(enc, dec, mode, rank)
    mine = vdist.shard_batch(full, rank, world, p["maxQuesCount"])
    eng = Engine(p)
    eng.set_math_mode(mode)
    eng.set_parameters(init_parameters(p, seed=3))
    eng.set_training(2)                      # training graph, dropout off: masks are indexed per local shard
    vdist.attach_engine(eng, rank, world)
    eng.zero_grad()
    loss = eng.forward_backward(Batch(mine))
    eng.clamp_adam_step(1e-3)
    w = eng.get_parameters()
    g = eng.get_gradients()                  # all-reduced, scaled, clamped
    gathered = vdist.gather_ranks(np.asarray([loss], dtype=np.float64), rank, world)
    if rank == 0:
        out.put((w, g, gathered))
    eng.close()
    dist.destroy_process_group()


# mode 1 = fp32 (small shapes, CUDA-core kernels), 0 = TF32, 2 = F16: tensor-core kernels, option stream overlapped, and the
# bucketed gradient all-reduce overlapped with the backward pass (the benched schedule)
@pytest.mark.parametrize("enc,dec,mode", [("mn-att-ques-im-hist", "disc", 1), ("lf-ques", "gen", 1), ("mn-att-ques-im-hist", "disc", 2),
                                          ("mn-att-ques-im-hist", "disc", 0), ("hrea-ques-im-hist", "gen", 0),
                                          ("lf-ques-im-hist", "disc", 2)])
def test_two_gpus_match_one(enc, dec, mode):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from visdial_b200 import Batch, Engine, init_parameters
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, enc, dec, mode, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    w2, g2, losses = q.get(timeout=300)
    for pr in procs:
        pr.join(timeout=60)
        assert pr.exitcode == 0
    p, full = _case(enc, dec, mode, 0)
    eng = Engine(p)
    eng.set_math_mode(mode)
    eng.set_parameters(init_parameters(p, seed=3))
    eng.set_training(2)
    eng.zero_grad()
    loss1 = eng.forward_backward(Batch(full))
    eng.clamp_adam_step(1e-3)
    w1, g1 = eng.get_parameters(), eng.get_gradients()
    eng.close()
    if dec == "disc":                        # mean criterion: global loss = mean of the equal-size shard losses
        assert float(np.mean(losses)) == pytest.approx(loss1, rel=1e-5)
    else:                                    # sum criterion: global loss = sum of the shard losses
        assert float(np.sum(losses)) == pytest.approx(loss1, rel=1e-5)
    scale = max(float(np.abs(g1).max()), 1e-30)
    # fp32: reduction order only.  Tensor-core modes: the 1-GPU and 2-GPU runs tile the option rows differently and the
    # fp16 BPTT picks its power-of-two scale per rank, so operand rounding differs at the 1e-3 level (stated TF32 class)
    tol = 1e-5 if mode == 1 else 5e-3
    assert float(np.abs(g2 - g1).max()) < tol * scale + 1e-7
    if mode == 1:
        assert float(np.abs(w2 - w1).max()) < 0.02 * 1e-3        # Adam steps are ~lr: compare in units of lr
