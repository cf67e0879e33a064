"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.npz by running the UNMODIFIED reference.

Run in the authoring container only (needs /root/reference):

    python oracle/gen_golden.py

Every vector below is produced by the reference's own classes (RGCN.RGCNBlockLayer, utils.*,
Aggregator.RGCNAggregator, model.RENet) imported through oracle/ref_loader.py over the pure-torch DGL
stand-in, on CPU fp32, dropout 0.  The fixtures are small and committed; the GPU box (which has no
/root/reference) checks both oracle/restate.py and the CUDA path against them.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')


def det_params(shapes, seed):
    """Deterministic parameter values, reproducible without the reference: for each name in sorted
    order, uniform(-a, a) with a = sqrt(6/(fan_in+fan_out)) * sqrt(2) (xavier/relu-gain-like);
    1-D tensors uniform(-0.05, 0.05)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name in sorted(shapes):
        shp = tuple(shapes[name])
        if len(shp) == 1:
            out[name] = (torch.rand(shp, generator=g) - 0.5) * 0.1
        else:
            a = (6.0 / (shp[0] + shp[1])) ** 0.5 * 2 ** 0.5
            out[name] = (torch.rand(shp, generator=g) * 2 - 1) * a
    return out


def shim_graph(ns, n, src, dst, type_s, type_o, norm=None):
    g = ns.dgl.DGLGraph()
    g.add_nodes(n)
    g.add_edges(src, dst)
    if norm is None:
        norm = ns.utils.comp_deg_norm(g)
    g.ndata['norm'] = torch.as_tensor(norm, dtype=torch.float32).view(-1, 1)
    g.edata['type_s'] = torch.as_tensor(type_s, dtype=torch.long)
    g.edata['type_o'] = torch.as_tensor(type_o, dtype=torch.long)
    return g


def run_layer(ns, case):
    """Reference RGCNBlockLayer forward + backward on one case dict (numpy inputs)."""
    import torch.nn.functional as F
    d_in, d_out, nb, R2 = case['d_in'], case['d_out'], case['nb'], case['R2']
    layer = ns.RGCN.RGCNBlockLayer(d_in, d_out, R2, nb, activation=F.relu if case['relu'] else None,
                                   self_loop=case['self_loop'], dropout=0.0)
    with torch.no_grad():
        layer.weight.copy_(torch.from_numpy(case['W']))
        if case['self_loop']:
            layer.loop_weight.copy_(torch.from_numpy(case['Wloop']))
    g = shim_graph(ns, case['N'], case['src'], case['dst'], case['type_s'], case['type_o'], case.get('norm'))
    H = torch.from_numpy(case['H']).clone().requires_grad_(True)
    g.ndata['h'] = H
    layer(g, bool(case['reverse']))
    out = g.ndata['h']
    res = {'out': out.detach().numpy().copy(), 'norm': g.ndata['norm'].view(-1).numpy().copy()}
    if case['N'] > 0:
        G = torch.from_numpy(case['G'])
        (out * G).sum().backward()
        res['dH'] = H.grad.numpy().copy()
        res['dW'] = layer.weight.grad.numpy().copy()
        if case['self_loop']:
            res['dWloop'] = layer.loop_weight.grad.numpy().copy()
    return res


def layer_cases():
    rng = np.random.RandomState(1234)
    cases = []

    def mk(name, N, src, dst, ts, to, d, nb, R2, relu, reverse, self_loop=True, int_w=False, norm=None):
        si = d // nb
        if int_w:
            W = rng.randint(-2, 3, size=(R2, nb * si * si)).astype(np.float32)
            Wl = rng.randint(-1, 2, size=(d, d)).astype(np.float32)
            H = rng.randint(-3, 4, size=(N, d)).astype(np.float32)
        else:
            W = (rng.rand(R2, nb * si * si).astype(np.float32) * 2 - 1) * 0.3
            Wl = (rng.rand(d, d).astype(np.float32) * 2 - 1) * 0.2
            H = rng.randn(N, d).astype(np.float32)
        c = dict(name=name, N=N, src=np.asarray(src, np.int64), dst=np.asarray(dst, np.int64),
                 type_s=np.asarray(ts, np.int64), type_o=np.asarray(to, np.int64), d_in=d, d_out=d, nb=nb, R2=R2,
                 relu=int(relu), reverse=int(reverse), self_loop=bool(self_loop), W=W, Wloop=Wl, H=H,
                 G=rng.randn(N, d).astype(np.float32))
        if norm is not None:
            c['norm'] = np.asarray(norm, np.float32)
        cases.append(c)

    R = 2
    # (1) hand KAT: triples {(0,r0,1),(2,r1,1)} -> get_big_graph edge layout [s->o.., o->s..]
    mk('hand_kat', 3, [0, 2, 1, 1], [1, 1, 0, 2], [0, 1, 0 + R, 1 + R], [0 + R, 1 + R, 0, 1], 4, 2, 2 * R, False, False, int_w=True)
    # (2) duplicate edge: same triple twice -> in-degree 2, message counted twice
    mk('dup_edge', 2, [0, 0, 1, 1], [1, 1, 0, 0], [0, 0, R, R], [R, R, 0, 0], 4, 2, 2 * R, False, False, int_w=True)
    # (3) reverse selects type_o
    mk('reverse', 3, [0, 2, 1, 1], [1, 1, 0, 2], [0, 1, 0 + R, 1 + R], [0 + R, 1 + R, 0, 1], 4, 2, 2 * R, True, True, int_w=True)
    # (4) explicit norm different from 1/in-degree (sub-graph norm is whatever the caller recomputed)
    mk('custom_norm', 3, [0, 2, 1], [1, 1, 0], [0, 1, 2], [2, 3, 0], 4, 2, 4, True, False, norm=[0.5, 0.25, 1.0])
    # (5) isolated nodes (no in-edge) + relu + no self loop
    mk('isolated_noloop', 5, [0, 1], [1, 0], [0, 1], [1, 0], 8, 4, 2, True, False, self_loop=False)
    # (6) random differential, RE-Net's real shape d=200 nb=100
    for N, E, R2, relu, rev in ((1, 3, 8, True, False), (33, 200, 16, True, True), (300, 2500, 32, False, False),
                                (257, 4000, 256, True, True)):
        src = rng.randint(0, N, E); dst = rng.randint(0, N, E)
        if N == 257:   # heavy-degree node (in-degree > 128) and empty relations
            dst[:300] = 7
        ts = rng.randint(0, R2, E); to = rng.randint(0, R2, E)
        mk('rand_N%d_E%d' % (N, E), N, src, dst, ts, to, 200, 100, R2, relu, rev)
    # (7) small generic shape with si=so=3
    src = rng.randint(0, 20, 90); dst = rng.randint(0, 20, 90)
    mk('generic_d12_nb4', 20, src, dst, rng.randint(0, 6, 90), rng.randint(0, 6, 90), 12, 4, 6, True, False)
    return cases


def gen_layers(ns):
    blob = {}
    names = []
    with ref_loader.cpu_patches():
        for c in layer_cases():
            res = run_layer(ns, c)
            names.append(c['name'])
            for k, v in c.items():
                if k != 'name':
                    blob['%s/%s' % (c['name'], k)] = np.asarray(v)
            for k, v in res.items():
                blob['%s/ref_%s' % (c['name'], k)] = v
        # (8) zero-edge graph: DGL 0.4 skips the reduce, only apply (h*norm) runs
        g = shim_graph(ns, 4, [], [], [], [])
        import torch.nn.functional as F
        layer = ns.RGCN.RGCNBlockLayer(4, 4, 2, 2, activation=F.relu, self_loop=True, dropout=0.0)
        H = torch.arange(16, dtype=torch.float32).view(4, 4) - 6
        g.ndata['h'] = H.clone()
        layer(g, False)
        blob['zero_edge/H'] = H.numpy(); blob['zero_edge/W'] = layer.weight.detach().numpy()
        blob['zero_edge/Wloop'] = layer.loop_weight.detach().numpy()
        blob['zero_edge/ref_out'] = g.ndata['h'].detach().numpy()
    blob['names'] = np.asarray(names)
    np.savez_compressed(os.path.join(OUT, 'layer_cases.npz'), **blob)
    print('layer_cases.npz: %d cases' % len(names))


SAMPLE_ROWS = 32


def random_layer_cases():
    """Four random graphs for RE-Net's layer shape (d=200, nb=100, 32 relation types), rebuilt identically without the
    reference: structure from one RandomState(0) stream, features and weights from seeded torch generators."""
    rng = np.random.RandomState(0)
    cases = []
    for k in range(4):
        N, E, R2 = int(rng.randint(1, 400)), int(rng.randint(1, 3000)), 32
        src, dst = rng.randint(0, N, E), rng.randint(0, N, E)
        ty = rng.randint(0, R2, E)
        P = det_params({'weight': (R2, 4 * 100), 'loop_weight': (200, 200)}, 100 + k)
        H = torch.randn(N, 200, generator=torch.Generator().manual_seed(200 + k))
        cases.append(dict(N=N, src=src, dst=dst, ty=ty, H=H, W=P['weight'], Wloop=P['loop_weight']))
    return cases


def gen_random_layers(ns):
    """Reference RGCNBlockLayer (relu, self-loop) on random_layer_cases(): its degree norm, and of each output the
    max-abs, the float64 row and column sums and SAMPLE_ROWS seeded rows (all rows together would be 0.7 MB)."""
    import torch.nn.functional as F
    blob = {}
    with ref_loader.cpu_patches():
        for k, c in enumerate(random_layer_cases()):
            layer = ns.RGCN.RGCNBlockLayer(200, 200, 32, 100, activation=F.relu, self_loop=True)
            with torch.no_grad():
                layer.weight.copy_(c['W'])
                layer.loop_weight.copy_(c['Wloop'])
            g = ns.dgl.DGLGraph(); g.add_nodes(c['N']); g.add_edges(c['src'], c['dst'])
            g.ndata['norm'] = ns.utils.comp_deg_norm(g).view(-1, 1)
            g.edata['type_s'] = torch.as_tensor(c['ty']); g.edata['type_o'] = torch.as_tensor(c['ty'])
            g.ndata['h'] = c['H'].clone()
            layer(g, False)
            out = g.ndata['h'].detach().numpy()
            rows = np.sort(np.random.RandomState(k).choice(c['N'], min(c['N'], SAMPLE_ROWS), replace=False))
            blob.update({'%d/norm' % k: g.ndata['norm'].view(-1).numpy(), '%d/rows' % k: rows, '%d/out_rows' % k: out[rows],
                         '%d/absmax' % k: np.abs(out).max(), '%d/rowsum' % k: out.astype(np.float64).sum(1),
                         '%d/colsum' % k: out.astype(np.float64).sum(0)})
    np.savez_compressed(os.path.join(OUT, 'reference_random_layers.npz'), **blob)
    print('reference_random_layers.npz: %d cases' % len(random_layer_cases()))


RENET_SHAPES = lambda num_e, h, R, nb: {  # noqa: E731
    'rel_embeds': (2 * R, h), 'ent_embeds': (num_e, h),
    'encoder.weight_ih_l0': (3 * h, 4 * h), 'encoder.weight_hh_l0': (3 * h, h),
    'encoder.bias_ih_l0': (3 * h,), 'encoder.bias_hh_l0': (3 * h,),
    'encoder_r.weight_ih_l0': (3 * h, 3 * h), 'encoder_r.weight_hh_l0': (3 * h, h),
    'encoder_r.bias_ih_l0': (3 * h,), 'encoder_r.bias_hh_l0': (3 * h,),
    'aggregator.rgcn1.weight': (2 * R, nb * (h // nb) ** 2), 'aggregator.rgcn1.loop_weight': (h, h),
    'aggregator.rgcn2.weight': (2 * R, nb * (h // nb) ** 2), 'aggregator.rgcn2.loop_weight': (h, h),
    'linear.weight': (num_e, 3 * h), 'linear.bias': (num_e,),
    'linear_r.weight': (R, 2 * h), 'linear_r.bias': (R,),
}


def det_global_emb(times, h, seed):
    g = torch.Generator().manual_seed(seed)
    return {int(t): 0.1 * torch.randn(1, 1, h, generator=g) for t in sorted(int(x) for x in times)}


def run_renet(ns, quads, num_e, R, h, nb, sel, seed, hist_builder):
    """Reference RENet.forward for both directions on the samples ``sel`` of ``quads``."""
    with ref_loader.cpu_patches():
        gd = {}
        for t in np.unique(quads[:, 3]):
            gd[int(t)] = ns.utils.get_big_graph(quads[quads[:, 3] == t][:, :3], R)
        S, ST, O, OT = hist_builder(quads)
        m = ns.model.RENet(num_e, h, R, dropout=0, model=0, seq_len=10, num_k=10)
        if nb != 100:
            m.aggregator = ns.Aggregator.RGCNAggregator(h, 0, num_e, R, nb, 0, 10)
        params = det_params(RENET_SHAPES(num_e, h, R, nb), seed)
        m.load_state_dict(params, strict=True)
        m.global_emb = det_global_emb(np.unique(quads[:, 3]), h, seed + 1)
        batch = torch.from_numpy(quads[sel]).long()
        sh = ([S[i] for i in sel], [ST[i] for i in sel])
        oh = ([O[i] for i in sel], [OT[i] for i in sel])
        res = {}
        captured = {}
        orig_enc, orig_encr = m.encoder.forward, m.encoder_r.forward

        def cap(name, orig):
            def f(x, *a, **k):
                captured[name] = x
                return orig(x, *a, **k)
            return f
        m.encoder.forward = cap('p4', orig_enc)
        m.encoder_r.forward = cap('p3', orig_encr)
        for subj in (True, False):
            m.zero_grad()
            loss = m(batch, sh, oh, gd, subject=subj)
            loss.backward()
            tag = 'subj' if subj else 'obj'
            res[tag + '/loss'] = np.float64(loss.item())
            res[tag + '/x4_sum'] = captured['p4'].data.detach().double().sum(0).numpy()     # column sums of the packed inputs
            res[tag + '/x3_sum'] = captured['p3'].data.detach().double().sum(0).numpy()
            res[tag + '/x4_head'] = captured['p4'].data[:16].detach().numpy().copy()
            res[tag + '/batch_sizes'] = captured['p4'].batch_sizes.numpy().copy()
            with torch.no_grad():
                _, s_h = orig_enc(captured['p4'])
                _, s_q = orig_encr(captured['p3'])
            res[tag + '/s_h'] = s_h.view(-1, h).numpy().copy()
            res[tag + '/s_q'] = s_q.view(-1, h).numpy().copy()
            for k, p in m.named_parameters():
                if p.numel() > 20000 and p.dim() == 2:
                    # large: store the norm and the two 1-D marginals instead of the full gradient
                    res['%s/grad_norm/%s' % (tag, k)] = np.float64(p.grad.double().norm().item())
                    res['%s/grad_rowsum/%s' % (tag, k)] = p.grad.double().sum(1).numpy()
                    res['%s/grad_colsum/%s' % (tag, k)] = p.grad.double().sum(0).numpy()
                else:
                    res['%s/grad/%s' % (tag, k)] = p.grad.numpy().copy()
    return res


def gen_renet_tiny(ns):
    sys.path.insert(0, ROOT)
    from oracle import restate
    rng = np.random.RandomState(7)
    num_e, R, T, h, nb = 50, 6, 14, 8, 4
    quads = []
    for t in range(T):
        n = rng.randint(20, 40)
        s = rng.zipf(1.4, n) % num_e
        o = rng.randint(0, num_e, n)
        r = rng.randint(0, R, n)
        quads += [[a, b, c, t * 24] for a, b, c in zip(s, r, o)]
    quads = np.asarray(quads, dtype=np.int64)
    sel = np.arange(len(quads) - 48, len(quads))
    res = run_renet(ns, quads, num_e, R, h, nb, sel, 11, lambda q: restate.build_history(q, num_e))
    res.update(quads=quads.astype(np.int32), sel=sel, num_e=num_e, R=R, h=h, nb=nb, seed=11)
    np.savez_compressed(os.path.join(OUT, 'renet_tiny.npz'), **res)
    print('renet_tiny.npz: loss', res['subj/loss'], res['obj/loss'])


def gen_renet_icews18_slice(ns):
    """A real ICEWS18 slice: the first 13 timestamps of the reference's train.txt, batch = 192 samples
    of the last two of them, h=200 / num_bases=100 (the real model shape)."""
    from oracle import restate
    q = np.loadtxt(os.path.join(ref_loader.REFERENCE_DIR, 'data', 'ICEWS18', 'train.txt'), dtype=np.int64)[:, :4]
    ts = np.unique(q[:, 3])[:13]
    quads = q[q[:, 3] <= ts[-1]]
    num_e, R, h, nb = 23033, 256, 200, 100
    cand = np.flatnonzero(quads[:, 3] >= ts[-2])
    sel = np.random.RandomState(999).permutation(cand)[:192]
    res = run_renet(ns, quads, num_e, R, h, nb, sel, 5, lambda qq: restate.build_history(qq, num_e))
    res.update(quads=quads.astype(np.int32), sel=sel, num_e=num_e, R=R, h=h, nb=nb, seed=5)
    np.savez_compressed(os.path.join(OUT, 'renet_icews18_slice.npz'), **res)
    print('renet_icews18_slice.npz: loss', res['subj/loss'], res['obj/loss'], 'quads', len(quads))


def gen_renet_eval_tiny(ns):
    """Test-time path (model.py:107-446) of the reference on the tiny TKG: init_history, filtered + raw ranks at the
    first test timestamp (no roll-over), then the roll-over to the second test timestamp (sampling from a stub global
    model, predicted graph, history roll) and the ranks after it."""
    from oracle import restate
    from oracle.stub_global import StubGlobalModel
    blob = np.load(os.path.join(OUT, 'renet_tiny.npz'))
    quads = blob['quads'].astype(np.int64)
    num_e, R, h, nb, seed = int(blob['num_e']), int(blob['R']), int(blob['h']), int(blob['nb']), 21
    times = np.unique(quads[:, 3])
    t_valid, t_test = times[-4], times[-2]
    S, ST, O, OT = restate.build_history(quads, num_e)
    split = lambda lo, hi: np.flatnonzero((quads[:, 3] >= lo) & (quads[:, 3] < hi))   # noqa: E731
    tr, va, te = split(0, t_valid), split(t_valid, t_test), split(t_test, times[-1] + 1)
    pick = lambda L, idx: [L[i] for i in idx]                                           # noqa: E731
    with ref_loader.cpu_patches():
        gd = {int(t): ns.utils.get_big_graph(quads[quads[:, 3] == t][:, :3], R) for t in times}
        m = ns.model.RENet(num_e, h, R, dropout=0, model=0, seq_len=10, num_k=5)
        m.aggregator = ns.Aggregator.RGCNAggregator(h, 0, num_e, R, nb, 0, 10)
        m.load_state_dict(det_params(RENET_SHAPES(num_e, h, R, nb), seed), strict=True)
        m.eval()
        m.global_emb = det_global_emb(times, h, seed + 1)
        m.graph_dict = gd
        m.init_history(quads[tr], (pick(S, tr), pick(ST, tr)), (pick(O, tr), pick(OT, tr)),
                       quads[va], (pick(S, va), pick(ST, va)), (pick(O, va), pick(OT, va)),
                       quads[te], (pick(S, te), pick(ST, te)), (pick(O, te), pick(OT, te)))
        res = {'hist_len_s': np.array([len(x) for x in m.s_hist_test]), 'hist_len_o': np.array([len(x) for x in m.o_hist_test]),
               'hist_last_t_s': np.array([x[-1] if len(x) else -1 for x in m.s_hist_test_t])}
        m.latest_time = torch.tensor(int(t_test))
        gm = StubGlobalModel(num_e, h, seed + 2)
        allq = torch.from_numpy(quads)
        torch.manual_seed(1234)
        out = {k: [] for k in ('raw', 'filt', 'loss', 'sub_pred', 'ob_pred')}
        with torch.no_grad():
            for i in te:
                trip = torch.from_numpy(quads[i])
                sh, oh = (S[i], ST[i]), (O[i], OT[i])
                rolled = int(trip[3]) != int(m.latest_time)
                fr, loss = m.evaluate_filter(trip, sh, oh, gm, allq)
                if rolled:
                    res['rolled_at'] = np.int64(i)
                    res['after_len_s'] = np.array([len(x) for x in m.s_hist_test])
                    res['after_len_o'] = np.array([len(x) for x in m.o_hist_test])
                    rows = [np.concatenate([[e], r]) for e in range(num_e) if len(m.s_hist_test_t[e]) and m.s_hist_test_t[e][-1] == int(t_test)
                            and len(m.s_hist_test[e]) for r in np.asarray(m.s_hist_test[e][-1]).reshape(-1, 2)]
                    res['after_new_s_rows'] = np.unique(np.asarray(rows, dtype=np.int64).reshape(-1, 3), axis=0)
                    g = m.graph_dict[int(t_test)]
                    res['pred_graph_nodes'] = np.sort(g.ndata['id'].view(-1).numpy())
                    res['pred_graph_num_edges'] = np.int64(g.number_of_edges())
                rr, _ = m.evaluate(trip, sh, oh, gm)
                _, sp, op = m.predict(trip, sh, oh, gm)
                out['raw'].append(rr); out['filt'].append(fr); out['loss'].append(loss.item())
                out['sub_pred'].append(sp.numpy().copy()); out['ob_pred'].append(op.numpy().copy())
    res.update({k: np.asarray(v) for k, v in out.items()})
    res.update(tr=tr, va=va, te=te, seed=seed, num_k=5, gm_calls=np.asarray(gm.calls, dtype=np.int64))
    np.savez_compressed(os.path.join(OUT, 'renet_eval_tiny.npz'), **res)
    print('renet_eval_tiny.npz: %d test triples, rolled at %s, mean filt rank %.2f, calls %d' % (
        len(te), res.get('rolled_at'), res['filt'].mean(), len(gm.calls)))


def gen_graph_kats(ns):
    """utils.get_big_graph / make_subgraph / get_sorted_s_r_embed_rgcn structure on a tiny stream."""
    from oracle import restate
    rng = np.random.RandomState(3)
    num_e, R = 12, 3
    quads = np.asarray([[rng.randint(num_e), rng.randint(R), rng.randint(num_e), t * 24]
                        for t in range(6) for _ in range(9)], dtype=np.int64)
    blob = {'quads': quads.astype(np.int32), 'num_e': num_e, 'R': R}
    with ref_loader.cpu_patches():
        for t in np.unique(quads[:, 3]):
            g = ns.utils.get_big_graph(quads[quads[:, 3] == t][:, :3], R)
            blob['g%d/id' % t] = g.ndata['id'].view(-1).numpy()
            blob['g%d/norm' % t] = g.ndata['norm'].view(-1).numpy()
            blob['g%d/src' % t] = g._src.numpy(); blob['g%d/dst' % t] = g._dst.numpy()
            blob['g%d/type_s' % t] = g.edata['type_s'].numpy(); blob['g%d/type_o' % t] = g.edata['type_o'].numpy()
        # make_subgraph: nodes {all ids of graph at t=24 except the first}
        g = ns.utils.get_big_graph(quads[quads[:, 3] == 24][:, :3], R)
        nodes = g.ndata['id'].view(-1).tolist()[1:]
        sg = ns.utils.make_subgraph(g, nodes)
        blob['sub/nodes'] = np.asarray(nodes)
        blob['sub/id'] = sg.ndata['id'].view(-1).numpy(); blob['sub/norm'] = sg.ndata['norm'].view(-1).numpy()
        blob['sub/src'] = sg._src.numpy(); blob['sub/dst'] = sg._dst.numpy()
        blob['sub/type_s'] = sg.edata['type_s'].numpy()
    S, ST, O, OT = restate.build_history(quads, num_e)
    # history structure (validated against the reference's preprocessing loop semantics in the tests)
    blob['hist_len_s'] = np.asarray([len(x) for x in S]); blob['hist_len_o'] = np.asarray([len(x) for x in O])
    np.savez_compressed(os.path.join(OUT, 'graph_kats.npz'), **blob)
    print('graph_kats.npz')


def _ref_model(ns, quads, num_e, R, h, nb, seed):
    gd = {}
    for t in np.unique(quads[:, 3]):
        gd[int(t)] = ns.utils.get_big_graph(quads[quads[:, 3] == t][:, :3], R)
    m = ns.model.RENet(num_e, h, R, dropout=0, model=0, seq_len=10, num_k=10)
    if nb != 100:
        m.aggregator = ns.Aggregator.RGCNAggregator(h, 0, num_e, R, nb, 0, 10)
    m.load_state_dict(det_params(RENET_SHAPES(num_e, h, R, nb), seed), strict=True)
    m.global_emb = det_global_emb(np.unique(quads[:, 3]), h, seed + 1)
    return m, gd


def gen_aggregator_predict(ns):
    """RGCNAggregator.forward (ELEMENT-wise packed inputs), .predict_batch and .predict (Aggregator.py:124-237) run by
    the unmodified reference: on the tiny stream (h=8, every element stored) and on the real ICEWS18 slice (h=200:
    predict fully; predict_batch called the way model.py:172-191 calls it -- num_rels copies of one history -- of which
    the rows of copies 0, 1 and R-1 and the column sums of all rows are stored)."""
    from oracle import restate
    tiny = np.load(os.path.join(OUT, 'renet_tiny.npz'))
    slc = np.load(os.path.join(OUT, 'renet_icews18_slice.npz'))
    blob = {}
    for tag, b in (('tiny', tiny), ('slice', slc)):
        quads = b['quads'].astype(np.int64)
        num_e, R, h, nb, seed = int(b['num_e']), int(b['R']), int(b['h']), int(b['nb']), int(b['seed'])
        sel = b['sel']
        with ref_loader.cpu_patches():
            m, gd = _ref_model(ns, quads, num_e, R, h, nb, seed)
            S, ST, O, OT = restate.build_history(quads, num_e)
            batch = torch.from_numpy(quads[sel]).long()
            for d, subj in (('subj', True), ('obj', False)):
                hist = ([S[i] for i in sel], [ST[i] for i in sel]) if subj else ([O[i] for i in sel], [OT[i] for i in sel])
                rel = m.rel_embeds[:R] if subj else m.rel_embeds[R:]
                s = batch[:, 0] if subj else batch[:, 2]
                r = batch[:, 1]
                with torch.no_grad():
                    if tag == 'tiny':
                        p4, p3 = m.aggregator(hist, s, r, m.ent_embeds, rel, gd, m.global_emb, not subj)
                        blob['%s/%s/fwd_x4' % (tag, d)] = p4.data.numpy().copy()
                        blob['%s/%s/fwd_x3' % (tag, d)] = p3.data.numpy().copy()
                        blob['%s/%s/fwd_bs' % (tag, d)] = p4.batch_sizes.numpy().copy()
                        # predict_batch on different histories whose lengths already descend (it never sorts, utils.py:251)
                        lens = np.asarray([len(x) for x in hist[0]])
                        order = [int(i) for i in np.argsort(-lens, kind='stable') if lens[i] > 0][:12]
                        hb = ([hist[0][i] for i in order], [hist[1][i] for i in order])
                        q4, q3 = m.aggregator.predict_batch(hb, s[order], r[order], m.ent_embeds, rel, gd, m.global_emb, not subj)
                        blob['%s/%s/pb_order' % (tag, d)] = np.asarray(order)
                        blob['%s/%s/pb_x4' % (tag, d)] = q4.data.numpy().copy()
                        blob['%s/%s/pb_x3' % (tag, d)] = q3.data.numpy().copy()
                        blob['%s/%s/pb_bs' % (tag, d)] = q4.batch_sizes.numpy().copy()
                    # the sample with the longest history: predict, and predict_batch as pred_r_rank2 calls it
                    lens = np.asarray([len(x) for x in hist[0]])
                    k = int(np.argmax(lens))
                    blob['%s/%s/k' % (tag, d)] = np.int64(k)
                    inp, inp_r = m.aggregator.predict((hist[0][k], hist[1][k]), s[k], r[k], m.ent_embeds, rel, gd,
                                                      m.global_emb, not subj)
                    blob['%s/%s/pred_x4' % (tag, d)] = inp.numpy().copy()
                    blob['%s/%s/pred_x3' % (tag, d)] = inp_r.numpy().copy()
                    ss = s[k].repeat(R)
                    rr = torch.arange(R)
                    q4, q3 = m.aggregator.predict_batch(([hist[0][k]] * R, [hist[1][k]] * R), ss, rr, m.ent_embeds, rel, gd,
                                                        m.global_emb, not subj)
                    L = int(lens[k])
                    rows = np.asarray([t * R + q for t in range(L) for q in (0, 1, R - 1)])
                    blob['%s/%s/rank_rows' % (tag, d)] = rows
                    blob['%s/%s/rank_x4' % (tag, d)] = q4.data[rows].numpy().copy()
                    blob['%s/%s/rank_x3' % (tag, d)] = q3.data[rows].numpy().copy()
                    blob['%s/%s/rank_x4_sum' % (tag, d)] = q4.data.double().sum(0).numpy()
                    blob['%s/%s/rank_bs' % (tag, d)] = q4.batch_sizes.numpy().copy()
    np.savez_compressed(os.path.join(OUT, 'aggregator_predict.npz'), **blob)
    print('aggregator_predict.npz:', len(blob), 'arrays')


def gen_global_tiny(ns):
    """RENet_global (global_model.py) run by the unmodified reference on the tiny stream: training loss + gradients for a
    batch of timestamps (both directions, max and mean pooling), predict() at one time, and get_global_emb() -- the
    vectors the hot path consumes as global_emb[t].  h = 200 because the reference hard-codes num_bases = 100."""
    tiny = np.load(os.path.join(OUT, 'renet_tiny.npz'))
    quads = tiny['quads'].astype(np.int64)
    num_e, R, h, seed = int(tiny['num_e']), int(tiny['R']), 200, 21
    times = np.unique(quads[:, 3])
    blob = {'h': h, 'seed': seed, 'times': times}
    with ref_loader.cpu_patches():
        gd = {}
        for t in times:
            gd[int(t)] = ns.utils.get_big_graph(quads[quads[:, 3] == t][:, :3], R)
        tps, tpo = ns.utils.get_true_distribution(quads, num_e)
        blob['true_prob_s'], blob['true_prob_o'] = tps, tpo
        for pool in (1, 0):
            m = ns.global_model.RENet_global(num_e, h, R, dropout=0, model=3, seq_len=10, num_k=10, maxpool=pool)
            shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
            m.load_state_dict(det_params(shapes, seed), strict=True)
            if pool == 1:
                blob['shapes_keys'] = np.asarray(sorted(shapes))
                blob['shapes_vals'] = np.asarray([list(shapes[k]) + [0] * (2 - len(shapes[k])) for k in sorted(shapes)])
            t_batch = torch.from_numpy(times[[5, 0, 12, 3, 13, 1]])
            sel = [5, 0, 12, 3, 13, 1]
            for subj in (True, False):
                m.zero_grad()
                loss = m(t_batch, torch.from_numpy(tps[sel]), torch.from_numpy(tpo[sel]), gd, subject=subj)
                loss.backward()
                tag = 'pool%d/%s' % (pool, 'subj' if subj else 'obj')
                blob[tag + '/loss'] = np.float64(loss.item())
                for k, p in m.named_parameters():
                    if p.grad is not None:
                        blob['%s/grad/%s' % (tag, k)] = p.grad.numpy().copy()
            with torch.no_grad():
                s_q, sub, prob = m.predict(int(times[7]), gd)
                blob['pool%d/pred_sq' % pool] = s_q.view(-1).numpy().copy()
                blob['pool%d/pred_sub' % pool] = sub.view(-1).numpy().copy()
                if pool == 1:
                    ge = m.get_global_emb(times, gd)
                    blob['pool1/global_emb_keys'] = np.asarray(sorted(ge))
                    blob['pool1/global_emb'] = np.stack([ge[k].view(-1).numpy() for k in sorted(ge)])
                    packed = m.aggregator(torch.from_numpy(times[[12, 5, 3]]), m.ent_embeds, gd, reverse=False)
                    blob['pool1/agg_packed'] = packed.data.numpy().copy()
                    blob['pool1/agg_bs'] = packed.batch_sizes.numpy().copy()
    blob['t_batch'] = np.asarray([5, 0, 12, 3, 13, 1])
    np.savez_compressed(os.path.join(OUT, 'global_tiny.npz'), **blob)
    print('global_tiny.npz: losses', blob['pool1/subj/loss'], blob['pool1/obj/loss'], blob['pool0/subj/loss'])


def gen_renet_eval_global(ns):
    """The reference's whole test flow with its OWN global model (test.py:41-150): RENet_global (deterministic parameters)
    produces global_emb for the training timestamps (pretrain.py:92) and drives the roll-over at test time; RENet
    (h = 200, num_bases = 100: the shape the CUDA fast path serves; the reference hard-codes 100 bases in the global
    aggregator) is evaluated with evaluate_filter over the test split of the tiny stream.  Stored: the global_emb table,
    every filtered rank, and MRR / MR / Hits@1/3/10 as test.py prints them."""
    from oracle import restate
    tiny = np.load(os.path.join(OUT, 'renet_tiny.npz'))
    quads = tiny['quads'].astype(np.int64)
    num_e, R, h, nb, seed = int(tiny['num_e']), int(tiny['R']), 200, 100, 31
    times = np.unique(quads[:, 3])
    t_valid, t_test = times[-4], times[-2]
    S, ST, O, OT = restate.build_history(quads, num_e)
    split = lambda lo, hi: np.flatnonzero((quads[:, 3] >= lo) & (quads[:, 3] < hi))   # noqa: E731
    tr, va, te = split(0, t_valid), split(t_valid, t_test), split(t_test, times[-1] + 1)
    pick = lambda L, idx: [L[i] for i in idx]                                           # noqa: E731
    with ref_loader.cpu_patches():
        gd = {int(t): ns.utils.get_big_graph(quads[quads[:, 3] == t][:, :3], R) for t in times}
        gm = ns.global_model.RENet_global(num_e, h, R, dropout=0, model=3, seq_len=10, num_k=5, maxpool=1)
        gshapes = {k: tuple(v.shape) for k, v in gm.state_dict().items()}
        gm.load_state_dict(det_params(gshapes, seed + 1), strict=True)
        gm.eval()
        m = ns.model.RENet(num_e, h, R, dropout=0, model=0, seq_len=10, num_k=5)
        m.load_state_dict(det_params(RENET_SHAPES(num_e, h, R, nb), seed), strict=True)
        m.eval()
        train_times = [int(t) for t in np.unique(quads[tr][:, 3])]
        with torch.no_grad():
            ge = gm.get_global_emb(train_times, gd)
        m.global_emb = ge
        res = {'global_emb_keys': np.asarray(sorted(ge)), 'global_emb': np.stack([ge[k].view(-1).numpy() for k in sorted(ge)])}
        m.graph_dict = gd
        m.init_history(quads[tr], (pick(S, tr), pick(ST, tr)), (pick(O, tr), pick(OT, tr)),
                       quads[va], (pick(S, va), pick(ST, va)), (pick(O, va), pick(OT, va)),
                       quads[te], (pick(S, te), pick(ST, te)), (pick(O, te), pick(OT, te)))
        for ee in range(num_e):                                     # test.py:100-106
            while len(m.s_hist_test[ee]) > 10:
                m.s_hist_test[ee].pop(0); m.s_hist_test_t[ee].pop(0)
            while len(m.o_hist_test[ee]) > 10:
                m.o_hist_test[ee].pop(0); m.o_hist_test_t[ee].pop(0)
        m.latest_time = torch.tensor(int(t_test))
        allq = torch.from_numpy(quads)
        torch.manual_seed(4321)
        ranks, losses = [], []
        with torch.no_grad():
            for i in te:                                            # test.py:113-136
                fr, loss = m.evaluate_filter(torch.from_numpy(quads[i]), (S[i], ST[i]), (O[i], OT[i]), gm, allq)
                ranks.append(fr); losses.append(loss.item())
    ranks = np.concatenate(ranks)
    res.update(ranks=ranks, loss=np.asarray(losses), mrr=np.mean(1.0 / ranks), mr=np.mean(ranks),
               hits=np.asarray([np.mean(ranks <= k) for k in (1, 3, 10)]), tr=tr, va=va, te=te, seed=seed, h=h, nb=nb, num_k=5,
               gshape_keys=np.asarray(sorted(gshapes)),
               gshape_vals=np.asarray([list(gshapes[k]) + [0] * (2 - len(gshapes[k])) for k in sorted(gshapes)]))
    np.savez_compressed(os.path.join(OUT, 'renet_eval_global.npz'), **res)
    print('renet_eval_global.npz: %d ranks, MRR %.6f MR %.3f Hits@1/3/10 %s' % (len(ranks), res['mrr'], res['mr'], res['hits']))


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    ns = ref_loader.load()
    torch.manual_seed(0)
    gen_layers(ns)
    gen_graph_kats(ns)
    gen_renet_tiny(ns)
    gen_renet_icews18_slice(ns)
    gen_renet_eval_tiny(ns)
    gen_aggregator_predict(ns)
    gen_global_tiny(ns)
    gen_renet_eval_global(ns)
    gen_random_layers(ns)
