"""-m gpu, needs >= 2 GPUs (skipped otherwise): the data-parallel training step over NCCL (SURVEY.md section 8e, config C4).

Two ranks each run the train-mode forward + hand-written backward on THEIR utterances of one fixed batch, the flat gradient
bucket is all-reduced (SUM) by the product code (tacotron_b200/optim.py through Tacotron.train_step), then clip + Adam.
Rank 0 also computes both shards' gradients alone on its own GPU: because the loss is a sum over utterances
(models/tacotron.py:158-160) the all-reduced bucket must equal the sum of the two single-process gradients -- bit for bit
(one fp32 addition per element either way) -- and both ranks must end the step with identical parameters."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _case():
    from oracle import tacotron_oracle as O
    B, Tx, T = 4, 12, 6                                    # 2 utterances per rank
    cfg = O.OracleConfig(r=2, vocab_size=20)
    p = O.init_params(cfg, seed=1, trained_like=True)
    inp = O.synthetic_inputs(cfg, B, Tx, T, seed=0, ragged=True)
    enc_m, dec_m = O.dropout_masks(cfg, B, Tx, T, seed=2)
    sm = O.sched_mask(cfg, B, T, seed=3)
    return cfg, p, inp, enc_m, dec_m, sm


def _shard(inp, enc_m, dec_m, sm, lo, hi):
    gi = {k: v[lo:hi].contiguous().cuda() for k, v in inp.items()}
    em = tuple(m[lo:hi].contiguous().cuda() for m in enc_m)
    dm = tuple(m[:, lo:hi].contiguous().cuda() for m in dec_m)
    return gi, em, dm, sm[:, lo:hi].contiguous().cuda()


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    import torch.distributed as dist
    from tacotron_b200 import Config, Tacotron
    from tacotron_b200.models import ops
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    cfg_o, p, inp, enc_m, dec_m, sm = _case()
    per = inp["text"].shape[0] // world

    def model():
        m = Tacotron(Config(r=cfg_o.r, vocab_size=cfg_o.vocab_size, precision="fp32"), None, train=True)
        m.load_params(p)
        return m

    # ---- the data-parallel step ----
    m = model()
    gi, em, dm, smr = _shard(inp, enc_m, dec_m, sm, rank * per, (rank + 1) * per)
    m.train_step(gi, lr=1e-3, enc_drop_masks=em, dec_drop_masks=dm, sample_mask=smr)
    torch.cuda.synchronize()
    g_dp = m._opt.g.clone()                                # the all-reduced bucket
    flat = m.store.flat.clone()
    # both ranks hold the same parameters after the step
    other = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(other, flat)
    same_params = all(torch.equal(o, other[0]) for o in other)
    res = {"same_params": bool(same_params)}
    if rank == 0:
        # ---- single-process reference: both shards on this GPU, no collective ----
        tot = torch.zeros_like(g_dp)
        for r in range(world):
            mr = model()
            mr.dp = False
            gir, emr, dmr, smrr = _shard(inp, enc_m, dec_m, sm, r * per, (r + 1) * per)
            S = {}
            with ops.saving(S):
                mr.seq2seq_output, mr.output = mr.inference(gir, True, enc_drop_masks=emr, dec_drop_masks=dmr, sample_mask=smrr)
            S.update(text=gir["text"], text_length=gir["text_length"], mel=gir["mel"], stft=gir["stft"])
            S["post/out"] = mr.output
            mr.backward(S)
            torch.cuda.synchronize()
            tot += mr._opt.g
        res["max_abs_diff"] = float((g_dp - tot).abs().max())
        res["ref_max"] = float(tot.abs().max())
        res["bit_equal"] = bool(torch.equal(g_dp, tot))
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_dp2_nccl_gradient_equals_single_process_sum():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert out[0]["same_params"] and out[1]["same_params"]
    # world size 2: NCCL's sum is one fp32 addition per element, like the local reference
    assert out[0]["max_abs_diff"] <= 1e-6 * out[0]["ref_max"], dict(out[0])
