"""GPU, 2 ranks over NCCL (skipped with fewer than 2 GPUs): ModuleNetTrainer.train_step on sharded
halves of a batch — forward, backward, the ONE all-reduce of the flat gradient (+ loss), per-tensor
clip, Adam, weight re-pack — ends with the weights and losses of one rank stepping on the full
batch (SURVEY.md §8e; exp_clevr/train_clevr_rl_gt_layout.py:119-139 for the step itself). Also the
eval path: each rank's pool evaluates its shard, the gathered scores equal the full-batch scores."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
N, H, W, D, T, C, STEPS = 32, 10, 15, 512, 10, 28, 3


def _case():
    from n2nmn_b200 import synth, weights as wts
    from n2nmn_b200.assembler import Assembler
    feat, word_vecs = synth.make_inputs(N, H, W, D, T, seed=91)
    Wt = wts.init_weights('clevr', H, W, D, C, seed=4, bias_std=0.1)
    asm = Assembler(synth.vocab_file('clevr'))
    tokens = [np.ascontiguousarray(synth.expert_mix_tokens(asm, N, T)[
        :, np.random.RandomState(s).permutation(N)]) for s in range(STEPS)]
    labels = [np.random.RandomState(40 + s).randint(0, C, size=N) for s in range(STEPS)]
    return feat, word_vecs, Wt, asm, tokens, labels


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from n2nmn_b200.executor import LayoutExecutor
    from n2nmn_b200.trainer import ModuleNetTrainer
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    solo = dist.new_group([0])           # every rank must take part in creating it
    feat, word_vecs, Wt, asm, tokens, labels = _case()
    per = N // world
    sl = slice(rank * per, (rank + 1) * per)
    f = torch.from_numpy(feat[sl].copy()).to(dev)
    w = torch.from_numpy(np.ascontiguousarray(word_vecs[:, sl])).to(dev)
    ex = LayoutExecutor('clevr', f, w, C, asm, weights=Wt, max_batch=N, max_T=T)
    tr = ModuleNetTrainer(ex)            # default group: all ranks
    losses = []
    for s in range(STEPS):
        out_s = tr.train_step(f, w, np.ascontiguousarray(tokens[s][:, sl]), labels[s][sl])
        losses.append(out_s['avg_sample_loss'])
    eval_scores, _ = ex.forward_device(f, w, np.ascontiguousarray(tokens[0][:, sl]))
    gathered = [torch.empty_like(eval_scores) for _ in range(world)]
    dist.all_gather(gathered, eval_scores)
    res = {'w': tr.w.cpu().numpy(), 'losses': losses, 'eval': torch.cat(gathered).cpu().numpy()}
    if rank == 0:                        # the same steps on the full batch, one rank, no collective
        ff, ww = torch.from_numpy(feat).to(dev), torch.from_numpy(word_vecs).to(dev)
        ex1 = LayoutExecutor('clevr', ff, ww, C, asm, weights=Wt, max_batch=N, max_T=T)
        tr1 = ModuleNetTrainer(ex1, process_group=solo)
        l1 = [tr1.train_step(ff, ww, tokens[s], labels[s])['avg_sample_loss'] for s in range(STEPS)]
        e1, _ = ex1.forward_device(ff, ww, tokens[0])
        res.update(w1=tr1.w.cpu().numpy(), losses1=l1, eval1=e1.cpu().numpy())
        np.save(out, res, allow_pickle=True)
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_train_steps_match_one_rank_on_the_full_batch(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]; s.close()
    out = str(tmp_path / 'r0.npy')
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    r = np.load(out, allow_pickle=True).item()
    print('losses 2 ranks', r['losses'], 'one rank', r['losses1'],
          'max |dw|', float(np.max(np.abs(r['w'] - r['w1']))))
    np.testing.assert_allclose(r['losses'], r['losses1'], rtol=0, atol=2e-6)
    np.testing.assert_allclose(r['w'], r['w1'], rtol=0, atol=1e-6)
    # eval after the steps: shards gathered == full batch (weights agree to 1e-6)
    np.testing.assert_allclose(r['eval'], r['eval1'], rtol=0, atol=2e-4)
