"""-m gpu: the training step (reference train.py:136-143) on the CUDA kernels -- native clip+Adam kernels against
torch.optim.Adam, the flat-buffer trainer against an ordinary torch training loop, gradient parity between the device
batcher and the all-host batcher (ADVICE r1: backward on a device-assembled batch), and the 2-rank NCCL data-parallel
step against a single process that accumulates the same two shards."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _model(tkg, seed=0, dropout=0.0, dev=DEV):
    from renet_b200.model import RENet
    torch.manual_seed(seed)
    m = RENet(tkg.num_e, 200, tkg.num_r, dropout=dropout).to(dev)
    m.global_emb = {t: v.to(dev) for t, v in tkg.global_emb.items()}
    return m


def test_native_clip_adam_matches_torch():
    from renet_b200 import _lib
    L, P = _lib.lib(), _lib.ptr
    torch.manual_seed(0)
    n = 1_000_003                                     # not a multiple of 4: exercises the scalar tail
    n_alloc = n + 1
    p = torch.randn(n_alloc, device=DEV)[:n]
    ref = torch.nn.Parameter(p.clone())
    opt = torch.optim.Adam([ref], lr=1e-3, weight_decay=1e-5)
    m, v = torch.zeros(n_alloc, device=DEV)[:n], torch.zeros(n_alloc, device=DEV)[:n]
    sumsq = torch.zeros(1, device=DEV)
    ws = torch.empty(int(L.renet_grad_sumsq_workspace_bytes()) // 4, device=DEV)
    for step in range(1, 5):
        g = torch.randn(n, device=DEV) * (3.0 if step % 2 else 1e-4)         # clipped and un-clipped steps
        ref.grad = g.clone()
        total = torch.nn.utils.clip_grad_norm_([ref], 1.0)
        opt.step()
        _lib.check(L.renet_grad_sumsq(P(g), n, P(sumsq), 0, P(ws), ws.numel() * 4, _lib.stream()), 'sumsq')
        assert abs(float(sumsq.sqrt()) - float(total)) < 1e-4 * float(total)
        _lib.check(L.renet_adam_step(P(p), P(g), P(m), P(v), n, 1e-3, 0.9, 0.999, 1e-8, 1e-5, step, P(sumsq), 1.0, 1.0,
                                     _lib.stream()), 'adam')
        assert torch.allclose(p, ref.detach(), atol=2e-6, rtol=1e-5), (step, (p - ref.detach()).abs().max())


def test_trainer_equals_plain_torch_loop():
    """DataParallelTrainer (flat views, hooks, native optimiser; world 1) == backward + clip_grad_norm_ + torch Adam."""
    import copy
    from renet_b200 import _lib, synthetic
    from renet_b200.parallel import DataParallelTrainer
    tkg = synthetic.SyntheticTKG('icews18', seed=5, num_timestamps=14)
    m1 = _model(tkg).train()
    m2 = copy.deepcopy(m1)
    m2.aggregator._pack_token = _lib.new_pack_token()
    m2.global_emb = m1.global_emb
    tr = DataParallelTrainer(m1, lr=1e-3, weight_decay=1e-5, grad_norm=1.0)
    opt = torch.optim.Adam(m2.parameters(), lr=1e-3, weight_decay=1e-5)
    for i in range(3):
        q, sh, oh = tkg.batch(i, batch_size=96)
        batch = torch.from_numpy(q).to(DEV)
        l1 = tr.train_step(batch, sh, oh, tkg.graph_dict)
        l2 = m2(batch, sh, oh, tkg.graph_dict, subject=True) + m2(batch, sh, oh, tkg.graph_dict, subject=False)
        l2.backward()
        torch.nn.utils.clip_grad_norm_(m2.parameters(), 1.0)
        opt.step()
        opt.zero_grad()
        assert abs(float(l1) - float(l2)) < 1e-4 * abs(float(l2)), (i, float(l1), float(l2))
    for (k, a), b in zip(m1.named_parameters(), m2.parameters()):
        # Adam normalises the update to ~lr per element whatever the gradient's scale: compare against lr
        assert (a - b).abs().max() < 2e-4, (k, float((a - b).abs().max()))


def test_backward_on_device_assembled_batch_matches_host_batcher():
    """ADVICE r1 (high): backward_structs() used to run before the device batcher's asynchronous edge count was
    resolved.  Gradients through RENet.forward + backward must agree between the device batcher (default), the all-host
    C++ batcher and the numpy list path."""
    from renet_b200 import hoststore, synthetic
    tkg = synthetic.SyntheticTKG('icews18', seed=7, num_timestamps=16)
    gs = hoststore.GraphStore(tkg.graph_dict)
    hs_s = hoststore.HistoryStore(tkg.s_hist, tkg.s_hist_t, tkg.quads[:, 0], gs)
    hs_o = hoststore.HistoryStore(tkg.o_hist, tkg.o_hist_t, tkg.quads[:, 2], gs)
    sel = tkg.batch_indices(0, 256)
    q, sh, oh = tkg.batch(0, 256)
    batch = torch.from_numpy(q).to(DEV)
    m = _model(tkg).train()

    def grads(hist_s, hist_o, gd, device_edges):
        hoststore.DEVICE_EDGES = device_edges
        m.zero_grad(set_to_none=True)
        loss = m(batch, hist_s, hist_o, gd, subject=True) + m(batch, hist_s, hist_o, gd, subject=False)
        loss.backward()
        return float(loss), {k: p.grad.clone() for k, p in m.named_parameters()}
    try:
        l_ref, g_ref = grads(sh, oh, tkg.graph_dict, True)                          # numpy list path
        l_dev, g_dev = grads(hs_s.select(sel), hs_o.select(sel), gs, True)          # device batcher
        l_host, g_host = grads(hs_s.select(sel), hs_o.select(sel), gs, False)       # all-host C++ batcher
        l_lst, g_lst = grads(sh, oh, gs, True)                                      # lists + GraphStore (view_from_lists)
    finally:
        hoststore.DEVICE_EDGES = True
    for l, g, tag in ((l_dev, g_dev, 'device'), (l_host, g_host, 'host'), (l_lst, g_lst, 'lists+store')):
        assert abs(l - l_ref) < 1e-5 * abs(l_ref), tag
        for k in g_ref:
            scale = float(g_ref[k].abs().max()) + 1e-12
            assert float((g[k] - g_ref[k]).abs().max()) < 1e-4 * scale, (tag, k)


# ---- 2 ranks over NCCL -----------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(('127.0.0.1', 0)); p = s.getsockname()[1]; s.close()
    return p


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from renet_b200 import synthetic
    from renet_b200.parallel import DataParallelTrainer, shard_batch
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    tkg = synthetic.SyntheticTKG('icews18', seed=11, num_timestamps=14)
    m = _model(tkg, dev=dev).train()
    grads = {}

    def capture(tr):            # stands in for the optimiser: record the reduced gradient
        for k, p in m.named_parameters():
            grads[k] = p.grad.detach().clone().cpu()
    tr = DataParallelTrainer(m, grad_norm=1.0, bucket_bytes=8 << 20, optimizer_step=capture)
    q, sh, oh = tkg.batch(0, batch_size=192)
    bq, bs, bo, n_local = shard_batch(q, sh, oh, rank, world)
    loss = tr.train_step(torch.from_numpy(bq).to(dev), bs, bo, tkg.graph_dict)
    torch.save({'loss': float(loss), 'grads': grads, 'buckets': len(tr.buckets)}, os.path.join(out_dir, 'rank%d.pt' % rank))
    dist.barrier()
    dist.destroy_process_group()


def test_nccl_two_rank_gradients_equal_accumulated_shards(tmp_path):
    """Global batch 192 = 2 x 96 over NCCL: the all-reduced gradient on every rank == the average of the two shards'
    gradients computed by ONE process.  (Not the gradient of one 192-sample batched graph: RE-Net's induced sub-graphs
    depend on which samples share a batch, utils.py:149-170, so sharding changes the graphs themselves; data parallelism
    averages per-shard losses, exactly like running the reference on the shards.)"""
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    import torch.multiprocessing as mp
    from renet_b200 import synthetic
    from renet_b200.parallel import shard_batch
    world, port = 2, _free_port()
    mp.spawn(_dp_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    res = [torch.load(os.path.join(str(tmp_path), 'rank%d.pt' % r)) for r in range(world)]
    assert res[0]['buckets'] > 1
    tkg = synthetic.SyntheticTKG('icews18', seed=11, num_timestamps=14)
    m = _model(tkg).train()
    q, sh, oh = tkg.batch(0, batch_size=192)
    losses = []
    for r in range(world):
        bq, bs, bo, _ = shard_batch(q, sh, oh, r, world)
        b = torch.from_numpy(bq).to(DEV)
        l = m(b, bs, bo, tkg.graph_dict, subject=True) + m(b, bs, bo, tkg.graph_dict, subject=False)
        (l / world).backward()
        losses.append(float(l))
    for r in range(world):
        assert abs(res[r]['loss'] - losses[r]) < 1e-5 * abs(losses[r])
        for k, p in m.named_parameters():
            ref = p.grad.cpu()
            scale = float(ref.abs().max()) + 1e-12
            assert float((res[r]['grads'][k] - ref).abs().max()) < 1e-5 * scale + 1e-9, (r, k)
    for k in res[0]['grads']:
        assert torch.equal(res[0]['grads'][k], res[1]['grads'][k]), k       # replicas see the identical reduced gradient


def test_fused_gru_input_dropout_exact_given_the_mask_and_statistics():
    """Training with the reference's default dropout never leaves the CUDA kernels: the fused GRU applies the aggregator's
    input dropout (Aggregator.py:157-158) with Philox masks.  Given the masks (renet_dropout_mask regenerates exactly what
    the kernels use) forward AND backward equal the CPU oracle on the masked inputs; the keep rate is 1-p; p=0 is untouched."""
    from helpers import rel_err
    from oracle import restate
    from renet_b200 import _lib, synthetic, utils
    from renet_b200.gru import fused_gru
    L, P = _lib.lib(), _lib.ptr
    tkg = synthetic.SyntheticTKG('icews18', seed=3, num_timestamps=24)
    q, sh, oh = tkg.batch(0, batch_size=256)
    hb = utils.assemble_history_batch(sh[0], sh[1], q[:, 0], tkg.graph_dict, torch.device(DEV))
    torch.manual_seed(0)
    h, p, seed = 200, 0.5, 1234567
    S, Q, N = hb.S, hb.num_seq, hb.graph.N
    H2 = (torch.randn(N, h) * 0.5).requires_grad_(True)
    ent, rel = (torch.randn(tkg.num_e, h) * 0.3).requires_grad_(True), (torch.randn(tkg.num_r, h) * 0.3).requires_grad_(True)
    glob = (torch.randn(len(hb.times), h) * 0.1).requires_grad_(True)
    enc, enc_r = torch.nn.GRU(4 * h, h, batch_first=True), torch.nn.GRU(3 * h, h, batch_first=True)
    s_tem, r_tem = torch.from_numpy(q[:, 0][hb.s_idx]), torch.from_numpy(q[:, 1][hb.s_idx])
    # the masks the kernels will use
    m = torch.empty(S * 7 * h, device=DEV)
    _lib.check(L.renet_dropout_mask(seed, 0, m.numel(), p, P(m), _lib.stream()), 'mask')
    m4, m3 = m[:S * 4 * h].view(S, 4 * h).cpu(), m[S * 4 * h:].view(S, 3 * h).cpu()
    keep = float((m > 0).float().mean())
    assert abs(keep - (1 - p)) < 2e-3 and set(m.unique().tolist()) == {0.0, 2.0}
    # oracle on the masked inputs (sequence-major rows)
    X4, X3, perm, bs = restate.packed_inputs(H2, hb.readout.cpu().long(), hb.seq_len, s_tem, r_tem, ent, rel,
                                             glob[hb.row_glob.cpu().long()])
    ref4 = restate.gru_final_hidden_batched(X4 * m4, hb.seq_len, enc.weight_ih_l0, enc.weight_hh_l0, enc.bias_ih_l0, enc.bias_hh_l0)
    ref3 = restate.gru_final_hidden_batched(X3 * m3, hb.seq_len, enc_r.weight_ih_l0, enc_r.weight_hh_l0, enc_r.bias_ih_l0, enc_r.bias_hh_l0)
    G4, G3 = torch.randn(ref4.shape), torch.randn(ref3.shape)
    ((ref4 * G4).sum() + (ref3 * G3).sum()).backward()
    ref_grads = [t.grad.clone() for t in (H2, ent, rel, glob)] + [pp.grad.clone() for mm in (enc, enc_r) for pp in mm.parameters()]
    # CUDA side
    import copy
    encd, encrd = copy.deepcopy(enc).to(DEV), copy.deepcopy(enc_r).to(DEV)
    for mm in (encd, encrd):
        mm.zero_grad()
    leaves = [t.detach().to(DEV).requires_grad_(True) for t in (H2, ent, rel, glob)]
    hn4, hn3 = fused_gru(leaves[0], leaves[1], leaves[2], leaves[3], hb, s_tem[:Q].to(torch.int32).to(DEV),
                         r_tem[:Q].to(torch.int32).to(DEV), encd, encrd, p_drop=p, seed=seed)
    assert rel_err(hn4.detach().cpu().numpy(), ref4.detach().numpy()) < 1e-4
    assert rel_err(hn3.detach().cpu().numpy(), ref3.detach().numpy()) < 1e-4
    ((hn4 * G4.to(DEV)).sum() + (hn3 * G3.to(DEV)).sum()).backward()
    got = [t.grad for t in leaves] + [pp.grad for mm in (encd, encrd) for pp in mm.parameters()]
    names = ['H2', 'ent', 'rel', 'glob'] + ['%s.%s' % (a, b) for a in ('enc', 'enc_r') for b, _ in enc.named_parameters()]
    for a, b, nm in zip(got, ref_grads, names):
        assert rel_err(a.cpu().numpy(), b.numpy()) < 2e-4, nm
    # p = 0 goes through the split-projection path and is untouched by any of this
    with torch.no_grad():
        a4, _ = fused_gru(leaves[0], leaves[1], leaves[2], leaves[3], hb, s_tem[:Q].to(torch.int32).to(DEV),
                          r_tem[:Q].to(torch.int32).to(DEV), encd, encrd)
        r4 = restate.gru_final_hidden_batched(X4.detach(), hb.seq_len, enc.weight_ih_l0, enc.weight_hh_l0, enc.bias_ih_l0, enc.bias_hh_l0)
    assert rel_err(a4.cpu().numpy(), r4.detach().numpy()) < 1e-4


def test_default_training_config_runs_on_our_kernels_only():
    """--dropout 0.5 (reference train.py:211): one training step launches no cuDNN RNN kernel -- the GRU modules are
    parameter holders only -- and the loss is finite and decreases over a few steps."""
    from renet_b200 import synthetic
    from renet_b200.parallel import DataParallelTrainer
    tkg = synthetic.SyntheticTKG('icews18', seed=5, num_timestamps=14)
    m = _model(tkg, dropout=0.5).train()
    called = []
    for mod in (m.encoder, m.encoder_r):
        mod.register_forward_hook(lambda *a: called.append(1))
    tr = DataParallelTrainer(m, lr=1e-3, weight_decay=1e-5, grad_norm=1.0)
    torch.manual_seed(0)
    losses = []
    q, sh, oh = tkg.batch(0, batch_size=128)
    batch = torch.from_numpy(q).to(DEV)
    for i in range(6):
        losses.append(float(tr.train_step(batch, sh, oh, tkg.graph_dict)))
    assert not called, 'nn.GRU.forward (cuDNN) was used'
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses


@pytest.mark.parametrize('M,N,K', [(1024, 23033, 600), (1024, 256, 400), (37, 1001, 24), (300, 199, 8)])
def test_fused_decoder_cross_entropy_vs_torch_fp32(M, N, K):
    """renet_decoder_ce_fwd/_bwd (tcgen05 3xTF32 GEMM with fused logsumexp epilogue, recompute-based backward) against a
    plain PyTorch fp64 reference of the same op (model.py:89-91,97-100): loss and all three gradients, including class
    counts that are not multiples of 8 / 200 and a last column tile of 33 classes (ICEWS18: 23033)."""
    from renet_b200.decoder import decoder_cross_entropy
    torch.manual_seed(M + N)
    x = torch.randn(M, K, device=DEV) * 0.5
    w = torch.randn(N, K, device=DEV) * (1.0 / K ** 0.5)
    b = torch.randn(N, device=DEV) * 0.1
    tgt = torch.randint(0, N, (M,), device=DEV)
    tgt[0], tgt[-1] = N - 1, 0
    xr, wr, br = (t.double().requires_grad_(True) for t in (x, w, b))
    ref = torch.nn.functional.cross_entropy(torch.nn.functional.linear(xr, wr, br), tgt)
    (0.7 * ref).backward()
    xs, ws_, bs = (t.clone().requires_grad_(True) for t in (x, w, b))
    loss = decoder_cross_entropy(xs, ws_, bs, tgt)
    assert abs(float(loss) - float(ref)) < 1e-5 * abs(float(ref)), (float(loss), float(ref))
    (0.7 * loss).backward()
    for a, r, nm in ((xs.grad, xr.grad, 'dX'), (ws_.grad, wr.grad, 'dW'), (bs.grad, br.grad, 'db')):
        err = float((a.double() - r).abs().max() / r.abs().max())
        assert err < 1e-4, (nm, err)
