"""-m "not gpu": pins oracle/restate.py against the golden vectors produced by the UNMODIFIED reference
(oracle/gen_golden.py)."""
import numpy as np
import torch

from helpers import layer_case, load_npz, rel_err, t
from oracle import restate
from oracle.gen_golden import RENET_SHAPES, det_global_emb, det_params, random_layer_cases

TOL = 2e-6   # CPU fp32 vs CPU fp32, same math in a different summation order


def _run_restate(c):
    H = t(c['H']).clone().requires_grad_(True)
    W = t(c['W']).clone().requires_grad_(True)
    Wl = t(c['Wloop']).clone().requires_grad_(True) if bool(c['self_loop']) else None
    et = t(c['type_o'] if int(c['reverse']) else c['type_s'])
    out = restate.rgcn_block_layer(H, W, Wl, t(c['src']), t(c['dst']), et, t(c['ref_norm']), bool(c['relu']), int(c['nb']))
    return H, W, Wl, out


def test_layer_cases_forward_backward():
    blob = load_npz('layer_cases.npz')
    for name in blob['names']:
        c = layer_case(blob, str(name))
        H, W, Wl, out = _run_restate(c)
        assert rel_err(out.detach().numpy(), c['ref_out']) < TOL, name
        (out * t(c['G'])).sum().backward()
        assert rel_err(H.grad.numpy(), c['ref_dH']) < 1e-5, name
        assert rel_err(W.grad.numpy(), c['ref_dW']) < 1e-5, name
        if Wl is not None:
            assert rel_err(Wl.grad.numpy(), c['ref_dWloop']) < 1e-5, name
        out2 = restate.rgcn_block_layer_ref_ops(H.detach(), W.detach(), None if Wl is None else Wl.detach(),
                                                t(c['src']), t(c['dst']),
                                                t(c['type_o'] if int(c['reverse']) else c['type_s']),
                                                t(c['ref_norm']), bool(c['relu']), int(c['nb']))
        assert rel_err(out2.numpy(), c['ref_out']) < TOL, name


def test_hand_kat_is_hand_computable():
    """3 nodes, triples {(0,r0,1),(2,r1,1)}, h=4, nb=2, integer weights: check one row by hand."""
    c = layer_case(load_npz('layer_cases.npz'), 'hand_kat')
    H, W, Wl = c['H'], c['W'], c['Wloop']
    # node 1 receives 0->1 (type 0) and 2->1 (type 1); in-degree 2 -> norm 0.5
    def blk(h, w):
        w = w.reshape(2, 2, 2)
        return np.concatenate([h[0:2] @ w[0], h[2:4] @ w[1]])
    want = 0.5 * (blk(H[0], W[0]) + blk(H[2], W[1])) + H[1] @ Wl
    np.testing.assert_allclose(c['ref_out'][1], want, rtol=0, atol=1e-6)


def test_zero_edge_graph():
    blob = load_npz('layer_cases.npz')
    H, W, Wl = t(blob['zero_edge/H']), t(blob['zero_edge/W']), t(blob['zero_edge/Wloop'])
    e = torch.zeros(0, dtype=torch.long)
    out = restate.rgcn_block_layer(H, W, Wl, e, e, e, torch.ones(4), True, 2)
    assert rel_err(out.numpy(), blob['zero_edge/ref_out']) < TOL


def test_graph_kats():
    b = load_npz('graph_kats.npz')
    quads, R = b['quads'].astype(np.int64), int(b['R'])
    gd = restate.build_graph_dict(quads, R)
    for tt, g in gd.items():
        np.testing.assert_array_equal(g.id, b['g%d/id' % tt])
        np.testing.assert_array_equal(g.src, b['g%d/src' % tt])
        np.testing.assert_array_equal(g.dst, b['g%d/dst' % tt])
        np.testing.assert_array_equal(g.type_s, b['g%d/type_s' % tt])
        np.testing.assert_array_equal(g.type_o, b['g%d/type_o' % tt])
        np.testing.assert_allclose(g.norm, b['g%d/norm' % tt], rtol=0, atol=0)
    sg = restate.induced_subgraph(gd[24], b['sub/nodes'].tolist())
    np.testing.assert_array_equal(sg.id, b['sub/id'])
    np.testing.assert_array_equal(sg.src, b['sub/src'])
    np.testing.assert_array_equal(sg.dst, b['sub/dst'])
    np.testing.assert_array_equal(sg.type_s, b['sub/type_s'])
    np.testing.assert_allclose(sg.norm, b['sub/norm'], rtol=0, atol=0)
    S, ST, O, OT = restate.build_history(quads, int(b['num_e']))
    np.testing.assert_array_equal([len(x) for x in S], b['hist_len_s'])
    np.testing.assert_array_equal([len(x) for x in O], b['hist_len_o'])


def _renet_vs_golden(fname, grad_tol):
    b = load_npz(fname)
    quads = b['quads'].astype(np.int64)
    num_e, R, h, nb, seed = int(b['num_e']), int(b['R']), int(b['h']), int(b['nb']), int(b['seed'])
    sel = b['sel']
    P = {k: v.clone().requires_grad_(True) for k, v in det_params(RENET_SHAPES(num_e, h, R, nb), seed).items()}
    glob = det_global_emb(np.unique(quads[:, 3]), h, seed + 1)
    gd = restate.build_graph_dict(quads, R)
    S, ST, O, OT = restate.build_history(quads, num_e)
    for tag, subj, (Hs, Ht) in (('subj', True, (S, ST)), ('obj', False, (O, OT))):
        for p in P.values():
            p.grad = None
        out = restate.renet_forward(P, quads[sel], [Hs[i] for i in sel], [Ht[i] for i in sel], gd, glob, subj, R, nb)
        assert abs(out['loss'].item() - float(b[tag + '/loss'])) < 2e-5 * abs(float(b[tag + '/loss']))
        np.testing.assert_array_equal(out['batch_sizes'], b[tag + '/batch_sizes'])
        X4p = out['X4'][torch.as_tensor(out['perm'])]
        assert rel_err(X4p.detach().double().sum(0).numpy(), b[tag + '/x4_sum']) < 1e-5
        assert rel_err(out['X3'].detach().double().sum(0).numpy(), b[tag + '/x3_sum']) < 1e-5
        # equal-length ties may be ordered differently (model.py:81 sort is unstable): compare as sets of rows
        for key, ref in (('s_h', b[tag + '/s_h']), ('s_q', b[tag + '/s_q'])):
            got = out[key].detach().numpy()
            assert got.shape == ref.shape
            assert rel_err(np.sort(got, axis=0), np.sort(ref, axis=0)) < 1e-4
        out['loss'].backward()
        for k in P:
            if (tag + '/grad/' + k) in b.files:
                assert rel_err(P[k].grad.numpy(), b[tag + '/grad/' + k]) < grad_tol, (tag, k)
            else:
                g = P[k].grad.double()
                assert abs(g.norm().item() - float(b['%s/grad_norm/%s' % (tag, k)])) < grad_tol * max(1e-12, float(b['%s/grad_norm/%s' % (tag, k)])), (tag, k)
                # marginals, measured against the gradient's own scale (the class-sum of a softmax
                # gradient is pure cancellation, so a relative error on it would be meaningless)
                scale = float(b['%s/grad_norm/%s' % (tag, k)])
                for ax, nm in ((1, 'grad_rowsum'), (0, 'grad_colsum')):
                    diff = np.abs(g.sum(ax).numpy() - b['%s/%s/%s' % (tag, nm, k)]).max()
                    assert diff < 10 * grad_tol * scale, (tag, k, nm)


def test_renet_tiny_golden():
    _renet_vs_golden('renet_tiny.npz', 2e-5)


def test_renet_icews18_slice_golden():
    _renet_vs_golden('renet_icews18_slice.npz', 5e-5)


def test_packed_order_matches_torch():
    lens = [10, 10, 7, 3, 1]
    perm, bs = restate.packed_order(lens)
    x = torch.zeros(5, 10, 1)
    k = 0
    for i, l in enumerate(lens):
        for j in range(l):
            x[i, j, 0] = k
            k += 1
    p = torch.nn.utils.rnn.pack_padded_sequence(x, lens, batch_first=True)
    np.testing.assert_array_equal(p.batch_sizes.numpy(), bs)
    np.testing.assert_array_equal(p.data.view(-1).long().numpy(), perm)
    assert list(bs) == [5, 4, 4, 3, 3, 3, 3, 2, 2, 2]


def test_gru_restatement_matches_nn_gru():
    torch.manual_seed(0)
    lens = [10, 10, 7, 3, 1]
    gru = torch.nn.GRU(12, 5, batch_first=True)
    X = torch.randn(sum(lens), 12)
    pad = torch.zeros(len(lens), 10, 12)
    k = 0
    for i, l in enumerate(lens):
        pad[i, :l] = X[k:k + l]
        k += l
    _, hn = gru(torch.nn.utils.rnn.pack_padded_sequence(pad, lens, batch_first=True))
    a = restate.gru_final_hidden(X, lens, gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0)
    b_ = restate.gru_final_hidden_batched(X, lens, gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0)
    assert rel_err(a.detach().numpy(), hn[0].detach().numpy()) < 1e-6
    assert rel_err(b_.detach().numpy(), hn[0].detach().numpy()) < 1e-6


def test_restate_vs_reference_random_layers():
    """The reference's RGCNBlockLayer on four random graphs (tests/golden/reference_random_layers.npz): the stored rows
    element-wise, every other row and column through its sum, all against the max-abs of the reference's whole output."""
    b = load_npz('reference_random_layers.npz')
    for k, c in enumerate(random_layer_cases()):
        g = lambda key: b['%d/%s' % (k, key)]                                          # noqa: E731
        out = restate.rgcn_block_layer(c['H'], c['W'], c['Wloop'], t(c['src']), t(c['dst']), t(c['ty']), t(g('norm')),
                                       True, 100).numpy()
        scale = float(g('absmax'))
        assert abs(np.abs(out).max() - scale) < TOL * scale, k
        assert np.abs(out[g('rows')] - g('out_rows')).max() < TOL * scale, k
        assert np.abs(out.astype(np.float64).sum(1) - g('rowsum')).max() < out.shape[1] * TOL * scale, k
        assert np.abs(out.astype(np.float64).sum(0) - g('colsum')).max() < out.shape[0] * TOL * scale, k


def _canon(x):
    """rows in a canonical order (ties among equal history lengths may be ordered differently, model.py:81)"""
    x = np.asarray(x, dtype=np.float64)
    return x[np.lexsort(np.round(x[:, ::-1] * 1e3).T)] if len(x) else x


def test_restatement_packed_inputs_elementwise_vs_reference_aggregator():
    """oracle/restate.py's packed GRU inputs, ELEMENT-wise, against RGCNAggregator.forward of the unmodified reference
    (tests/golden/aggregator_predict.npz, tiny stream)."""
    from oracle.gen_golden import RENET_SHAPES, det_global_emb, det_params
    tiny, gold = load_npz('renet_tiny.npz'), load_npz('aggregator_predict.npz')
    quads = tiny['quads'].astype(np.int64)
    num_e, R, h, nb, seed = (int(tiny[k]) for k in ('num_e', 'R', 'h', 'nb', 'seed'))
    P = det_params(RENET_SHAPES(num_e, h, R, nb), seed)
    glob = det_global_emb(np.unique(quads[:, 3]), h, seed + 1)
    gd = restate.build_graph_dict(quads, R)
    S, ST, O, OT = restate.build_history(quads, num_e)
    sel = tiny['sel']
    for d, subj, H, HT in (('subj', True, S, ST), ('obj', False, O, OT)):
        out = restate.renet_forward(P, quads[sel], [H[i] for i in sel], [HT[i] for i in sel], gd, glob, subj, R, nb)
        perm = out['perm']
        np.testing.assert_array_equal(out['batch_sizes'], gold['tiny/%s/fwd_bs' % d])
        for ours, ref in ((out['X4'][perm], gold['tiny/%s/fwd_x4' % d]), (out['X3'][perm], gold['tiny/%s/fwd_x3' % d])):
            # time-major packing: step t owns rows [sum(bs[:t]), sum(bs[:t+1])); compare step by step, rows canonicalised
            o = 0
            for n in out['batch_sizes']:
                assert rel_err(_canon(ours[o:o + n].numpy()), _canon(ref[o:o + n])) < 2e-6
                o += int(n)
