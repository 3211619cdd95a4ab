"""CPU tests (`-m "not gpu"`): the C-ABI library loads and exports what include/se_b200.h declares, the host
layer (graph builders, schedules, plans, DP plumbing) matches the fixtures recorded from the reference."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
G = os.path.join(ROOT, 'tests', 'golden')


@pytest.fixture(scope='session')
def built_lib():
    from semantic_embeddings_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    return _lib


def test_library_exports_every_declared_symbol(built_lib):
    hdr = open(os.path.join(ROOT, 'include', 'se_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = set(re.findall(r'\b(se_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 30
    lib = built_lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(built_lib.exported_symbols()), declared ^ set(built_lib.exported_symbols())
    assert lib.se_version().decode().startswith('se_b200')


def test_product_path_has_no_oracle_or_cpu_fallback():
    pkg = os.path.join(ROOT, 'semantic_embeddings_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f
    from semantic_embeddings_b200 import _lib
    saved = _lib.LIB_PATH
    try:
        _lib.LIB_PATH = saved + '.missing'
        _lib._lib = None
        with pytest.raises(_lib.SeError):
            _lib.load()
    finally:
        _lib.LIB_PATH = saved
        _lib._lib = None


def test_same_padding():
    from semantic_embeddings_b200.graph import same_pad
    assert same_pad(32, 3, 1) == (1, 1, 32)
    assert same_pad(32, 3, 2) == (0, 1, 16)       # TF SAME is asymmetric for stride 2
    assert same_pad(32, 1, 2) == (0, 0, 16)
    assert same_pad(7, 3, 2) == (1, 1, 4)


@pytest.mark.parametrize('tag', ['simple', 'resnet-110-fc', 'resnet-110', 'resnet-32', 'wrn-28-10'])
def test_graph_builders_match_reference_layer_trace(tag):
    """Layer names, kernel sizes, strides, padding, bias, L2, BN hyper-parameters and output shapes of the product's
    graphs vs the trace recorded from the reference's own model builders (make_golden.py)."""
    from semantic_embeddings_b200 import utils
    with open(os.path.join(G, 'arch_%s.json' % tag)) as f:
        meta = json.load(f)
    g = utils.build_network(meta['dim'], meta['architecture'], input_channels=3)
    nodes = {n.name: n for n in g.nodes}
    convs = [t for t in meta['trace'] if t['class'] == 'Conv2D']
    assert len(convs) == sum(1 for n in g.nodes if n.op == 'conv')
    for t in convs:
        n = nodes[t['name']]
        assert n.attrs['k'] == t['kernel_size'][0] == t['kernel_size'][1]
        assert n.attrs['stride'] == t['strides'][0]
        assert n.attrs['use_bias'] == t['use_bias']
        assert list(n.output.shape) == t['out_shape'], (t['name'], n.output.shape, t['out_shape'])
        assert g.params[t['name'] + '/kernel'].l2 == t['l2']
        assert g.params[t['name'] + '/kernel'].init == t['kernel_initializer']
        assert n.attrs['relu'] == (t['activation'] == 'relu')
    bns = [t for t in meta['trace'] if t['class'] == 'BatchNormalization' and t['name'] in nodes]
    assert len(bns) == sum(1 for n in g.nodes if n.op == 'bn')
    for t in bns:
        n = nodes[t['name']]
        assert abs(n.attrs['momentum'] - t['momentum']) < 1e-12 and abs(n.attrs['eps'] - t['epsilon']) < 1e-12
        assert g.params[t['name'] + '/gamma'].init == t['gamma_initializer']
    for t in meta['trace']:
        if t['class'] == 'Dense' and t['name'] in nodes:
            assert nodes[t['name']].output.shape == (t['units'],)
            assert g.params[t['name'] + '/kernel'].l2 == t['l2']
    last = [t for t in meta['trace'] if t['class'] == 'Lambda'][0]
    assert list(g.output.shape) == last['out_shape']


def test_model_sizes_match_survey():
    from semantic_embeddings_b200 import utils
    g = utils.build_network(100, 'resnet-110-fc')
    assert sum(1 for n in g.nodes if n.op == 'conv') == 109
    assert abs(g.conv_macs_per_image() / 1e6 - 252.89) < 0.01          # SURVEY.md Appendix B
    g = utils.build_network(100, 'simple')
    assert abs(g.conv_macs_per_image() / 1e6 - 247.14) < 0.01
    g = utils.build_network(100, 'wrn-28-10')
    assert abs(g.conv_macs_per_image() / 1e6 - 5243.3) < 0.1
    assert abs(g.num_params() / 1e6 - 36.5) < 0.1
    g = utils.build_network(555, 'resnet-50')
    assert sum(1 for n in g.nodes if n.op == 'conv') == 53


def test_build_network_errors_like_reference():
    from semantic_embeddings_b200 import utils
    with pytest.raises(ValueError, match='Unknown network architecture'):
        utils.build_network(10, 'no-such-net')                          # utils.py:276
    with pytest.raises(NotImplementedError):
        utils.build_network(10, 'pyramidnet-272-200')
    with pytest.raises(ValueError, match='Unknown learning rate schedule'):
        utils.get_lr_schedule('nope', 1, 1, {})                         # utils.py:397-399


def test_sgdr_matches_reference_fixture():
    from semantic_embeddings_b200 import utils
    with open(os.path.join(G, 'sgdr_ref.json')) as f:
        ref = json.load(f)
    for tag in ('default', 'short'):
        cbs, num_epochs = utils.get_lr_schedule('SGDR', 50000, 128, dict(ref[tag]['args']))
        assert num_epochs == ref[tag]['num_epochs']
        s = cbs[0]
        s.on_train_begin()
        seq = []
        for ep in range(num_epochs):
            seq.append(s.lr)
            s.on_epoch_end(ep, {})
        np.testing.assert_allclose(seq, ref[tag]['lr'], rtol=1e-14)


def test_engine_builds_plans_without_a_gpu(built_lib):
    """device='cpu' allocates host tensors and builds the launch plans only (nothing is executed)."""
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    L = built_lib
    emb = np.load(os.path.join(G, 'class_matrices.npz'))['cifar100_embedding']
    for arch, cls_w in (('resnet-110-fc', 0.0), ('simple', 0.0), ('wrn-28-10', 0.1), ('resnet-110-fc', 0.1)):
        g = utils.build_network(100, arch)
        eng = Engine(g, 2, emb, cls_weight=cls_w, num_classes=100, device='cpu', use_cuda_graph=False)
        fwd, bwd = eng.plans['fwd'], eng.plans['bwd']
        nconv = sum(1 for n in eng.nodes if n.op in ('conv', 'dense'))
        assert sum(1 for o in fwd if o.opcode == L.OP_CONV_FWD) == nconv
        assert sum(1 for o in bwd if o.opcode == L.OP_CONV_WGRAD) == nconv
        # every conv but the stem (whose input is the image) needs a data gradient
        assert sum(1 for o in bwd if o.opcode == L.OP_CONV_DGRAD) == nconv - 1
        nbn = sum(1 for n in eng.nodes if n.op == 'bn')
        assert sum(1 for o in fwd if o.opcode == L.OP_BN_FWD_TRAIN) == nbn
        assert sum(1 for o in bwd if o.opcode == L.OP_BN_BWD) == nbn
        assert sum(1 for o in fwd if o.opcode == L.OP_HEAD) == 1
        assert sum(1 for o in bwd if o.opcode == L.OP_HEAD) == (1 if cls_w > 0 else 0)
        # L2 segments cover exactly the regularised kernels
        reg = sum(int(np.prod(p.shape)) for p in eng.pspecs.values() if p.trainable and p.l2 > 0)
        covered = sum(e - b for b, e, _ in eng.segments)
        assert reg <= covered <= reg + 4 * len(eng.pspecs)
        w = eng.get_weights() if False else None
    # plan-runner hints and the fused conv+BatchNorm op (engine.py _build_plans)
    g = utils.build_network(100, 'resnet-110-fc')
    eng = Engine(g, 2, emb, device='cpu', use_cuda_graph=False)
    fwd, bwd = eng.plans['fwd'], eng.plans['bwd']
    bn_bwd = [o for o in bwd if o.opcode == L.OP_BN_BWD]
    # i[4] = "inputs date from the forward pass, >= 24 launches ago" (prefetch before the grid dependency resolves):
    # set everywhere except for the last layers of the network, whose backward follows their forward closely
    assert bn_bwd[0].i[4] == 0 and bn_bwd[-1].i[4] == 1
    assert sum(o.i[4] for o in bn_bwd) >= len(bn_bwd) - 8
    first_early = next(k for k, o in enumerate(bn_bwd) if o.i[4])
    assert all(o.i[4] == 1 for o in bn_bwd[first_early:])
    assert not any(o.opcode == L.OP_CONV_BN_FWD for o in fwd)               # convolution and BatchNorm are separate launches
    # data-parallel plan: every gradient is exchanged exactly once, in buckets cut along the backward pass
    for arch, kw in (('resnet-110-fc', {}), ('simple', {}), ('wrn-28-10', {'cls_weight': 0.1})):
        e2 = Engine(utils.build_network(100, arch), 2, emb, device='cpu', use_cuda_graph=False, world_size=2, comm='torch', **kw)
        ar = [o for o in e2.plans['step_dp'] if o.opcode == L.OP_ALLREDUCE]
        assert len(ar) >= 3 and len(e2.plans['step_dp']) == len(e2.plans['step']) + len(ar)
        ranges = sorted((r[0], r[1]) for bucket in e2.bucket_ranges for r in bucket)
        assert ranges[0][0] == 0 and all(a[0] + a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
        assert ranges[-1][0] + ranges[-1][1] == e2.nparams
        # the last bucket (what cannot overlap with anything) is the smallest share of the buffer
        sizes = [sum(r[1] for r in bucket) for bucket in e2.bucket_ranges]
        assert sizes[-1] == min(sizes)
        pos = [k for k, o in enumerate(e2.plans['step_dp']) if o.opcode == L.OP_ALLREDUCE]
        last_bwd = max(k for k, o in enumerate(e2.plans['step_dp']) if o.opcode in (L.OP_CONV_WGRAD, L.OP_BN_BWD))
        first_opt = min(k for k, o in enumerate(e2.plans['step_dp']) if o.opcode == L.OP_SGD_PREPARE)
        assert pos[0] < last_bwd and last_bwd < pos[-1] < first_opt
    # --cls_base: the classifier head on the pooled features -- avg_pool then has two consumers, the head has none, so the
    # forward head op writes dz itself (no separate backward head op) and avg_pool's gradient is written (beta 0) by the
    # classifier branch, then accumulated into (beta 1) by the embedding layer's data gradient
    eb = Engine(utils.build_network(100, 'resnet-110-fc'), 2, emb, cls_weight=0.1, num_classes=100, device='cpu',
                use_cuda_graph=False, cls_base='avg_pool')
    assert eb.offsets['prob/kernel'][1] == (64, 100) and eb.offsets['cls_bn/gamma'][1] == (64,)
    assert sum(1 for o in eb.plans['bwd'] if o.opcode == L.OP_HEAD) == 0
    dg = [o for o in eb.plans['bwd'] if o.opcode == L.OP_CONV_DGRAD]
    assert dg[0].i[3] == 64 and dg[0].i[4] == 100 and dg[0].f[0] == 0.0        # prob: 64 -> 100, first write of its input gradient
    assert dg[1].i[3] == 64 and dg[1].i[4] == 100 and dg[1].f[0] == 1.0        # embedding: accumulates into avg_pool's gradient
    with pytest.raises(ValueError):
        Engine(utils.build_network(100, 'resnet-110-fc'), 2, emb, cls_weight=0.1, num_classes=100, device='cpu', cls_base='conv0')
    with pytest.raises(ValueError):
        Engine(utils.build_network(100, 'resnet-110-fc'), 2, emb, cls_weight=0.1, num_classes=100, device='cpu', cls_base='nope')
    # set_trainable: frozen runs + the L2 segments that remain partition the regularised range; thawing restores the plan
    n_opt = len(eng.plans['opt'])
    frozen = eng.set_trainable(lambda n: n.split('/')[0] == 'embedding')
    assert len(frozen) == len(eng.offsets) - 2 and eng.frozen_runs
    fr = sum(sz for _, sz in eng.frozen_runs)
    tr = sum((int(np.prod(eng.offsets[n][1])) + 3) // 4 * 4 for n in eng.offsets if n.split('/')[0] == 'embedding')
    assert fr + tr == eng.nparams
    segs = [(eng.seg_array[k].begin, eng.seg_array[k].end) for k in range(eng.n_active_segs)]
    assert all(not (b < o + sz and o < e) for b, e in segs for o, sz in eng.frozen_runs)      # no L2 term on frozen weights
    ek = eng.offsets['embedding/kernel']
    assert segs == [(ek[0], ek[0] + (int(np.prod(ek[1])) + 3) // 4 * 4)]
    assert len(eng.plans['opt']) == n_opt + len(eng.frozen_runs)
    assert all(o.opcode == L.OP_MEMSET and o.i[0] == 1 for o in list(eng.plans['opt'])[:len(eng.frozen_runs)])
    assert eng.set_trainable(None) == [] and len(eng.plans['opt']) == n_opt and eng.n_active_segs == len(eng.segments)
    # weight I/O round trip keeps Keras names and layouts
    g = utils.build_network(100, 'resnet-32')
    eng = Engine(g, 2, np.eye(64), device='cpu', use_cuda_graph=False)
    ws = g.init_weights(3)
    eng.set_weights(ws)
    v = eng._pview('res2-1x/kernel')
    assert tuple(v.shape) == (3, 3, 16, 32)
    np.testing.assert_array_equal(v.numpy(), ws['res2-1x/kernel'])
    with pytest.raises(KeyError):
        eng.set_weights({'nope/kernel': np.zeros(1)})
    with pytest.raises(ValueError):
        Engine(utils.build_network(100, 'resnet-110'), 2, emb, device='cpu')     # 64-d output vs 100-d classes


def test_shard_helpers():
    from semantic_embeddings_b200.parallel import shard_batch, shard_rows
    assert [shard_rows(50000, 8, r) for r in (0, 7)] == [(0, 6250), (43750, 6250)]
    assert [shard_rows(10, 4, r) for r in range(4)] == [(0, 3), (3, 3), (6, 3), (9, 1)]
    assert shard_rows(2, 4, 3) == (2, 0)
    assert [shard_batch(10, 4, r) for r in range(4)] == [(0, 2), (2, 2), (4, 2), (6, 4)]   # last tower takes the rest


_GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
from semantic_embeddings_b200.parallel import init_process_group, allreduce_gradients, broadcast_parameters, shard_rows
rank, world = init_process_group('gloo')
assert world == 2
flat = torch.arange(10, dtype=torch.float32) * (rank + 1)
allreduce_gradients(flat)
assert torch.equal(flat, torch.arange(10, dtype=torch.float32) * 3), flat
w = torch.full((5,), float(rank + 7))
broadcast_parameters([w], src=0)
assert torch.equal(w, torch.full((5,), 7.0))
# row-sharded retrieval: the shards tile [0, N) exactly once
r0, rows = shard_rows(1001, world, rank)
t = torch.zeros(1001); t[r0:r0 + rows] = 1
dist.all_reduce(t)
assert torch.equal(t, torch.ones(1001))
dist.destroy_process_group()
open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'rank' + str(rank) + '.ok'), 'w').write('ok')
'''


def test_data_parallel_plumbing_gloo_world2(tmp_path):
    script = tmp_path / 'worker.py'
    script.write_text(_GLOO_WORKER % {'root': ROOT})
    env = dict(os.environ, MASTER_ADDR='127.0.0.1')
    out = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node=2',
                          '--master-addr', '127.0.0.1', '--master-port', '29533', str(script)],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert (tmp_path / 'rank0.ok').exists() and (tmp_path / 'rank1.ok').exists(), out.stdout + out.stderr


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm): exactly one JSON line on stdout with
    the contract's keys; it times the oracle port of the reference training step on the host cores."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'images/s' and d['higher_is_better'] is True and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and 'sample' in d['cpu_baseline']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0 and d['e2e']['value'] == d['value']
    assert d['n_gpus'] == 1 and d['steps'] == 1


def test_class_hierarchy_restatement_matches_the_reference_tables(tmp_path):
    """semantic_embeddings_b200.class_hierarchy.ClassHierarchy (own implementation of class_hierarchy.py:7-208, :349-380)
    on the CIFAR-100 taxonomy: Wu-Palmer and LCS-height tables equal to the ones the reference's class produced
    (tests/golden/retrieval_ref.npz, make_golden.py), from a relation file in both orientations."""
    from semantic_embeddings_b200.class_hierarchy import ClassHierarchy, ideal_gains
    pc = np.load(os.path.join(GOLDEN, 'cifar_hierarchy.npz'))['parent_child']
    fx = np.load(os.path.join(GOLDEN, 'retrieval_ref.npz'))
    f1, f2 = tmp_path / 'pc.txt', tmp_path / 'isa.txt'
    f1.write_text('\n'.join('%d %d' % (p, c) for p, c in pc) + '\n\n')
    f2.write_text('\n'.join('%d %d' % (c, p) for p, c in pc) + '\n')
    for h in (ClassHierarchy.from_file(str(f1), id_type=int), ClassHierarchy.from_file(str(f2), is_a_relations=True, id_type=int)):
        wup, lcsh = h.similarity_luts(list(range(100)))
        assert np.array_equal(wup, fx['wup_lut']) and np.array_equal(lcsh, fx['lcs_height_lut'])
        assert h.is_tree() and h.wup_similarity(3, 3) == 1.0 and h.lcs_height(5, 5) == 0.0
        assert h.lcs(0, 0) == 0 and h.shortest_path_length(7, 7) == 0
    # ideal gains = cumsum of the sorted similarities of the whole database (class_hierarchy.py:268,280)
    labels = fx['labels'].astype(np.int32)
    bw, bl = ideal_gains(labels, wup, lcsh, len(labels))
    for c in (0, 17, 99):
        np.testing.assert_allclose(bw[c], np.cumsum(np.sort(wup[c, labels])[::-1]), rtol=0, atol=1e-12)
        np.testing.assert_allclose(bl[c], np.cumsum(np.sort(1.0 - lcsh[c, labels])[::-1]), rtol=0, atol=1e-12)
    with pytest.raises(ValueError):
        ClassHierarchy({1: [2], 2: [1]}, {2: [1], 1: [2]})          # a cycle


def test_cli_scripts_parse_their_reference_flags():
    """Both drop-in scripts import from the repo (never from /root/reference), accept the reference's flags
    (learn_image_embeddings.py:57-94, evaluate_retrieval.py:157-173) and reject malformed booleans like the reference."""
    import argparse
    import importlib
    lie = importlib.import_module('learn_image_embeddings')
    er = importlib.import_module('evaluate_retrieval')
    assert os.path.dirname(os.path.abspath(lie.__file__)) == ROOT and os.path.dirname(os.path.abspath(er.__file__)) == ROOT
    assert lie.get_data_generator.__module__ == 'semantic_embeddings_b200.datasets'
    a = lie.build_parser().parse_args(['--dataset', 'CIFAR-100', '--data_root', '/x', '--embedding', 'e.pickle', '--loss',
                                       'softmax_corr', '--max_decay', '0.1', '--top_k_acc', '5', '10', '--snapshot_best',
                                       '--sgdr_max_lr', '0.05', '--gpus', '8'])
    assert a.loss == 'softmax_corr' and a.top_k_acc == [5, 10] and a.snapshot_best == 'val_loss' and a.arith == 'tf32x3'
    assert a.batch_size == 100 and a.clipgrad == 10.0 and a.architecture == 'simple' and a.lr_schedule == 'SGDR'
    assert er.str2bool('T') is True and er.str2bool('no') is False
    with pytest.raises(argparse.ArgumentTypeError):
        er.str2bool('maybe')
    assert er.METRICS[4] == 'AHP (WUP)' and er.METRICS[-1] == 'AP' and len(er.METRICS) == 11
    assert callable(er.pairwise_retrieval)


def test_augment_oracle_is_the_scipy_transform_keras_delegates_to():
    """oracle/augment.py: shifts are scipy.ndimage.affine_transform(order=1, mode='nearest') per channel, flip afterwards,
    standardize with epsilon 1e-7; an integer shift is a plain roll with edge replication."""
    from oracle import augment as oaug
    rng = np.random.RandomState(1)
    x = rng.randint(0, 255, (8, 8, 3)).astype(np.float32)
    out = oaug.random_transform(x, 2.0, -1.0, False)          # out[h, w] = x[h + 2, w - 1], clamped
    hh = np.clip(np.arange(8) + 2, 0, 7)
    ww = np.clip(np.arange(8) - 1, 0, 7)
    assert np.allclose(out, x[hh][:, ww])
    assert np.allclose(oaug.random_transform(x, 0.0, 0.0, True), x[:, ::-1])
    half = oaug.random_transform(x, 0.5, 0.0, False)
    assert np.allclose(half[:-1], 0.5 * (x[:-1] + x[1:]), atol=1e-4) and np.allclose(half[-1], x[-1], atol=1e-4)
    mean, std = oaug.fit_statistics(np.stack([x, x + 1]))
    assert np.allclose(oaug.standardize(x, mean, std), (x - mean) / (std + 1e-7))


def test_finetune_weights_are_loaded_by_name_with_mismatches_skipped(built_lib, tmp_path):
    """learn_image_embeddings.load_weights_by_name = model.load_weights(by_name=True, skip_mismatch=True) (:185)."""
    import pickle
    import learn_image_embeddings as lie
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    eng = Engine(utils.build_network(64, 'simple'), 2, np.eye(64), device='cpu', use_cuda_graph=False)
    ws = utils.build_network(64, 'simple').init_weights(7)
    ws = {k: np.asarray(v, np.float32) + 1.0 for k, v in ws.items()}
    ws['embedding/kernel'] = np.zeros((ws['embedding/kernel'].shape[0], 100), np.float32)      # a 100-d head: does not fit
    ws['not_a_layer/kernel'] = np.zeros((3, 3), np.float32)
    for path in (tmp_path / 'dump.pickle', tmp_path / 'dump.npz'):
        if str(path).endswith('.npz'):
            np.savez(path, **ws)
        else:
            with open(path, 'wb') as f:
                pickle.dump({'architecture': 'simple', 'weights': ws}, f)
        loaded, skipped = lie.load_weights_by_name(eng, str(path))
        assert sorted(skipped) == ['embedding/kernel', 'not_a_layer/kernel'] and len(loaded) == len(ws) - 2
        name = loaded[0]
        np.testing.assert_array_equal(eng._pview(name).numpy(), ws[name])


def test_tensor_core_coverage_of_the_baseline_networks(built_lib):
    """se_conv2d_path (host-side planning, no GPU): which convolutions of the BASELINE architectures run on the tcgen05
    kernels in the benchmarked arithmetic, per direction (forward, backward data, weight gradient)."""
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.models import resnet50
    L = built_lib
    lib = L.load()

    def paths(graph, batch):
        out = {}
        for n in graph.nodes:
            if n.op != 'conv':
                continue
            h, w, cin = n.inputs[0].shape
            ho, wo, cout = n.output.shape
            a = n.attrs
            d = L.ConvDesc(batch, h, w, cin, cout, a['k'], a['k'], a['stride'], a['pad_t'], a['pad_l'], ho, wo)
            out[n.name] = (a['k'], a['stride'], cin) + tuple(lib.se_conv2d_path(d, L.SE_MODE_TF32X3, k) for k in range(3))
            assert all(lib.se_conv2d_path(d, L.SE_MODE_F32, k) == 0 for k in range(3))
        return out

    import bench
    cov = bench.tc_coverage(utils.build_network(100, 'resnet-110-fc', input_channels=3), 128, L.SE_MODE_TF32X3, L)
    assert cov == {'convolutions': 109, 'forward': 106, 'backward_data': 106, 'weight_gradient': 106}     # bench.py's config extra
    # config 4: every convolution of ResNet-50 at 224 x 224 except the 7x7 / 2 stem on 3 input channels
    r50 = paths(resnet50.ResNet50(555, input_shape=(224, 224, 3)), 32)
    assert len(r50) == 53 and [n for n, v in r50.items() if v[3:] != (1, 1, 1)] == ['conv1']
    assert sum(1 for v in r50.values() if v[0] == 1 and v[1] == 2) == 6             # the strided 1x1 layers are on it too
    # config 2 (headline): all 3x3 / stride 1 layers; the 3-channel stem and the two narrow 3x3 / stride 2 layers are fp32
    r110 = paths(utils.build_network(100, 'resnet-110-fc', input_channels=3), 128)
    off = {n: v for n, v in r110.items() if v[3:] != (1, 1, 1)}
    assert len(r110) == 109 and sorted(off) == ['conv0', 'res2-1x', 'res3-1x'] and all(v[3:] == (0, 0, 0) for v in off.values())
    # config 3: the wide 3x3 / stride 2 layers take the nine-tap tensor-core form in the backward pass, fp32 forward
    wrn = paths(utils.build_network(100, 'wrn-28-10', input_channels=3), 64)
    s2 = [v for v in wrn.values() if v[0] == 3 and v[1] == 2]
    assert len(s2) == 2 and all(v[3:] == (0, 1, 1) for v in s2)
    assert [n for n, v in wrn.items() if v[3:] == (0, 0, 0)] == [next(iter(wrn))]     # only the 3-channel stem


def test_bench_dump_outputs_samples_large_arrays_reproducibly(tmp_path):
    """bench.py --dump-outputs: arrays up to DUMP_MAX_ELEMENTS are written whole; a larger one as a sample at indices
    that depend only on its length, so that two runs (or two builds) write the same elements."""
    import bench
    n = bench.DUMP_MAX_ELEMENTS
    outs = {'small': np.arange(6, dtype=np.float64).reshape(2, 3), 'big': np.arange(n + 1000, dtype=np.float32)}
    for run in ('a', 'b'):
        bench.dump_outputs(outs, str(tmp_path / run))
    np.testing.assert_array_equal(np.load(str(tmp_path / 'a' / 'small.npy')), outs['small'])
    a, b = (np.load(str(tmp_path / run / 'big.npy')) for run in ('a', 'b'))
    assert a.dtype == np.float32 and a.shape == (n,) and np.array_equal(a, b)
    assert (np.diff(a) > 0).all() and a[-1] < n + 1000           # distinct elements, in index order
