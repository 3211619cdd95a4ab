"""GPU parity tests of whole training steps (engine + C-ABI library) against the CPU oracle, and of the
forward pass against the fixtures produced by the reference's own model-building code
(tests/golden/arch_*.npz, see make_golden.py).

North-star tolerance (BASELINE.json): embeddings and loss within 1e-4 relative of the reference
semantics in parity mode (SE_MODE_F32).  Gradients / updated weights are compared per tensor by
relative L2 error.
"""
import json
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(__file__), 'golden')
REPORT = os.path.join(os.path.dirname(os.path.dirname(__file__)), 'gpurun_out', 'parity_models.jsonl')


def report(name, **vals):
    try:
        os.makedirs(os.path.dirname(REPORT), exist_ok=True)
        with open(REPORT, 'a') as f:
            f.write(json.dumps(dict(test=name, **vals)) + '\n')
    except OSError:
        pass


def rel_l2(a, b):
    a = np.asarray(a, np.float64).ravel()
    b = np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def rel_max(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def class_matrix(key='cifar100'):
    return np.load(os.path.join(G, 'class_matrices.npz'))[key + '_embedding']


def oracle_weights_np(m, cls=None):
    w = {k: v.numpy().astype(np.float32) for k, v in m.params.items()}
    if cls is not None:
        w.update({k: v.numpy().astype(np.float32) for k, v in cls.params.items()})
    return w


def to_f32_exact(m, cls=None):
    """Round the oracle's float64 weights to float32 values so both sides start from identical numbers."""
    for v in m.params.values():
        v.copy_(v.float().double())
    if cls is not None:
        for v in cls.params.values():
            v.copy_(v.float().double())


@pytest.mark.parametrize('tag', ['simple', 'resnet-110-fc', 'resnet-110', 'resnet-32', 'wrn-28-10'])
def test_forward_matches_reference_graph_fixture(tag):
    """Engine forward (training-mode BN) vs the output of the reference's own graph code on the same weights."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    with open(os.path.join(G, 'arch_%s.json' % tag)) as f:
        meta = json.load(f)
    d = np.load(os.path.join(G, 'arch_%s.npz' % tag))
    s = meta['seeds']
    om = omodels.build_network(meta['dim'], meta['architecture'], input_channels=3, seed=s['build'])
    omodels.randomize(om, seed=s['randomize'])
    cls = None
    if meta['with_cls']:
        cls = otrain.ClsHead(meta['dim'], 100, seed=s['cls'])
        omodels.randomize(cls.params, seed=s['cls_rand'])
    graph = utils.build_network(meta['dim'], meta['architecture'], input_channels=3)
    B = meta['batch']
    emb = class_matrix('cifar100') if meta['dim'] == 100 else np.eye(meta['dim'])
    eng = Engine(graph, B, emb, loss='inv_corr', cls_weight=0.5 if cls is not None else 0.0, num_classes=100,
                 use_cuda_graph=False)
    eng.set_weights(oracle_weights_np(om, cls))
    eng.load_batch(torch.from_numpy(d['x'].astype(np.float32)), torch.zeros(B, dtype=torch.int64))
    eng._run('fwd')
    z = eng.act[graph.output.name].cpu().numpy()
    x_out = eng.act['head_out'].cpu().numpy()
    e_z, e_e = rel_max(z, d['z']), rel_max(x_out, d['emb'])
    e_p = 0.0
    if cls is not None:
        e_p = rel_max(eng.act['prob_out'].cpu().numpy(), d['prob'])
    report('forward_fixture', tag=tag, z=e_z, emb=e_e, prob=e_p)
    assert e_z < 1e-4 and e_e < 1e-4 and e_p < 1e-4, (e_z, e_e, e_p)


STEP_CASES = [
    # tag, arch, D/emb key, batch, loss, cls_weight, nesterov
    ('simple', 'simple', 'cifar100', 8, 'inv_corr', 0.0, False),
    ('resnet-32', 'resnet-32', None, 8, 'inv_corr', 0.0, False),
    ('resnet-110-fc', 'resnet-110-fc', 'cifar100', 8, 'inv_corr', 0.0, False),
    ('resnet-110-fc-cls', 'resnet-110-fc', 'cifar100', 8, 'inv_corr', 0.1, True),
    ('simple-mse', 'simple', 'cifar100', 6, 'mse', 0.0, False),
    ('wrn-28-10-cls', 'wrn-28-10', 'cifar100', 4, 'inv_corr', 0.1, False),
    # the same gate in the arithmetic the training path runs and bench.py measures (SE_MODE_TF32X3: tcgen05 tiles with
    # error compensation); the cases above run the fp32 FFMA kernels
    ('simple-x3', 'simple', 'cifar100', 8, 'inv_corr', 0.0, False, 2),
    ('resnet-110-fc-x3', 'resnet-110-fc', 'cifar100', 8, 'inv_corr', 0.0, False, 2),
    ('resnet-110-fc-cls-x3', 'resnet-110-fc', 'cifar100', 8, 'inv_corr', 0.1, True, 2),
    ('wrn-28-10-cls-x3', 'wrn-28-10', 'cifar100', 4, 'inv_corr', 0.1, False, 2),
]


def test_cls_base_inner_layer_step_matches_oracle():
    """--cls_base (learn_image_embeddings.py:34-40): the classifier head (relu -> BatchNorm -> Dense softmax) reads the
    64-d 'avg_pool' features instead of the embedding output; that tensor then has two consumers (the embedding layer and
    the classifier) whose gradients accumulate.  One step against the float64 oracle."""
    import copy
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('cifar100')
    C, D = emb.shape
    B, lr, cw = 8, 0.05, 0.1
    om = omodels.build_network(D, 'resnet-110-fc', input_channels=3, seed=21)
    omodels.randomize(om, seed=22)
    cls = otrain.ClsHead(64, C, seed=23)                     # on the 64-d pooled features
    omodels.randomize(cls.params, seed=24)
    to_f32_exact(om, cls)
    eng = Engine(utils.build_network(D, 'resnet-110-fc', input_channels=3), B, emb, cls_weight=cw, num_classes=C,
                 clipnorm=10.0, use_cuda_graph=False, cls_base='avg_pool')
    assert eng.offsets['prob/kernel'][1] == (64, C)
    eng.set_weights(oracle_weights_np(om, cls))
    vel = otrain.make_velocity(om, cls)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    g = torch.Generator().manual_seed(78)
    x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
    y = torch.randint(0, C, (B,), generator=g)
    om32, cls32 = copy.deepcopy(om), copy.deepcopy(cls)
    otrain.cast_model(om32, torch.float32, cls32)
    _, grads32, _ = otrain.train_step(om32, x, y, emb_t.float(), {k: v.float() for k, v in vel.items()}, lr, 'inv_corr', cls32, cw,
                                      False, 10.0, cls_base='avg_pool')
    obj, grads, norm = otrain.train_step(om, x.double(), y, emb_t, vel, lr, 'inv_corr', cls, cw, False, 10.0, cls_base='avg_pool')
    floor = max(_grad_errors({k: v.numpy() for k, v in grads32.items()}, grads, norm)[:2])
    eng.train_step(x, y, lr=lr)
    m = eng.metrics()
    e_loss = abs(m['loss'] - float(obj['embed_loss'].detach()))
    e_cls = abs(m['cls_loss'] - float(obj['cls_loss'].detach()))
    e_emb = rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].detach().numpy())
    e_prob = rel_max(eng.act['prob_out'].cpu().numpy(), obj['prob'].detach().numpy())
    gg, gw, name = _grad_errors(eng.get_grads(), grads, norm)
    report('cls_base_step', loss=e_loss, cls_loss=e_cls, emb=e_emb, prob=e_prob, grad_global=gg, worst=name, grad_floor_f32_oracle=floor)
    assert max(e_loss, e_cls, e_emb, e_prob) < 1e-4, (e_loss, e_cls, e_emb, e_prob)
    assert gg < max(2e-3, 5 * floor), (gg, floor)
    with pytest.raises(ValueError):
        Engine(utils.build_network(D, 'resnet-110-fc', input_channels=3), B, emb, cls_weight=cw, num_classes=C, cls_base='conv0')


def test_frozen_layers_step_matches_oracle():
    """--finetune_init phase (learn_image_embeddings.py:183-207): only the layers 'embedding' and 'prob' train.  Two steps
    against the float64 oracle restricted to those weights (Keras differentiates only with respect to trainable weights:
    clipping norm and L2 terms over them alone); every other parameter must stay bit-identical, BatchNorm moving
    statistics keep updating.  Then the thawed engine takes a full step again."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('cifar100')
    C, D = emb.shape
    B, lr, cw = 8, 0.05, 0.1
    om = omodels.build_network(D, 'resnet-110-fc', input_channels=3, seed=21)
    omodels.randomize(om, seed=22)
    cls = otrain.ClsHead(D, C, seed=23)
    omodels.randomize(cls.params, seed=24)
    to_f32_exact(om, cls)
    eng = Engine(utils.build_network(D, 'resnet-110-fc', input_channels=3), B, emb, cls_weight=cw, num_classes=C,
                 clipnorm=0.3, use_cuda_graph=True)                     # a clipping norm small enough to be active
    eng.set_weights(oracle_weights_np(om, cls))
    keep = lambda name: name.split('/')[0] in ('embedding', 'prob')
    frozen = eng.set_trainable(keep)
    assert frozen and all(not keep(n) for n in frozen) and len(frozen) + 4 == len(eng.offsets)
    om.trainable = [n for n in om.trainable if keep(n)]
    cls.trainable = [n for n in cls.trainable if keep(n)]
    vel = otrain.make_velocity(om, cls)
    w0 = eng.get_weights()
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    g = torch.Generator().manual_seed(77)
    for step in range(2):
        x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
        y = torch.randint(0, C, (B,), generator=g)
        obj, grads, norm = otrain.train_step(om, x.double(), y, emb_t, vel, lr, 'inv_corr', cls, cw, False, 0.3)
        eng.train_step(x, y, lr=lr)
        assert norm >= 0.3, norm                                        # the clip (over the trainable gradients only) is active
    w1 = eng.get_weights()
    ow = oracle_weights_np(om, cls)
    worst = 0.0
    for name in eng.offsets:
        if keep(name):
            worst = max(worst, rel_max(w1[name], ow[name]))
        else:
            assert np.array_equal(w1[name], w0[name]), name
    assert not np.array_equal(w1['bn0/moving_mean'], w0['bn0/moving_mean'])
    vel_e = eng.get_velocity()
    assert all(not vel_e[n].any() for n in frozen)
    report('frozen_step', trainable_weights=worst, frozen=len(frozen))
    assert worst < 1e-4, worst
    # thaw: every kernel moves again (the biases in front of a BatchNorm have gradients at rounding level: sum of a
    # normalised gradient -- their updates can vanish in fp32)
    assert eng.set_trainable(None) == []
    eng.train_step(x, y, lr=lr)
    w2 = eng.get_weights()
    assert all(not np.array_equal(w2[n], w1[n]) for n in eng.offsets if n.endswith('/kernel'))


class _relu_probe:
    """Context manager that replaces torch.relu while the oracle runs.  Without `flip` it records, per call, the
    element of smallest |pre-activation| (exact zeros excluded); with `flip=[(call, index), ...]` it inverts the
    mask of those elements (forward value changes by ~1e-7, the backward path through the element switches)."""

    def __init__(self, flip=None):
        self.flip = {}
        for call, idx in (flip or []):
            self.flip.setdefault(call, []).append(idx)
        self.records, self.calls = [], 0

    def __enter__(self):
        self._orig = torch.relu

        def patched(t):
            k = self.calls
            self.calls += 1
            mask = t > 0
            if k in self.flip:
                mask = mask.clone()
                flat = mask.view(-1)
                for idx in self.flip[k]:
                    flat[idx] = ~flat[idx]
            elif not self.flip:
                a = t.detach().abs().reshape(-1)
                a = torch.where(a == 0, torch.full_like(a, float('inf')), a)
                v, i = torch.topk(a, min(3, a.numel()), largest=False)
                self.records += [(float(vv), k, int(ii)) for vv, ii in zip(v, i)]
            return t * mask.to(t.dtype)

        torch.relu = patched
        return self

    def __exit__(self, *exc):
        torch.relu = self._orig
        return False

    def fragile(self, below=4e-6, at_most=4):
        """ReLU inputs so close to zero (activations are O(1)) that fp32 accumulation cannot resolve their sign."""
        return [(k, i) for v, k, i in sorted(self.records)[:at_most] if v < below]


def _grad_errors(eg, grads, norm):
    num = den = 0.0
    worst, worst_name = 0.0, ''
    for name, gr in grads.items():
        a = np.asarray(eg[name], np.float64)
        b = gr.numpy().astype(np.float64)
        num += float(((a - b) ** 2).sum())
        den += float((b ** 2).sum())
        r = rel_l2(a, b) if np.linalg.norm(b) > 1e-3 * norm else 0.0     # skip mathematically-zero grads (bias before BN)
        if r > worst:
            worst, worst_name = r, name
    return float(np.sqrt(num / den)), worst, worst_name


@pytest.mark.parametrize('case', STEP_CASES, ids=lambda c: c[0])
def test_two_training_steps_match_oracle(case):
    """Two optimizer steps against the float64 oracle.  Before each step the engine is given the oracle's
    weights / momentum / moving statistics (rounded to fp32 on both sides), so every step is a comparison on
    IDENTICAL inputs -- the north-star criterion -- while step 2 still exercises momentum and BN state.

    Embeddings, loss, regulariser, gradient norm: <= 1e-4 relative.  Gradients: ReLU networks are
    discontinuous in their pre-activations, so fp32 arithmetic legitimately flips a few masks relative to
    float64; the tolerance is therefore tied to the measured noise floor of the SAME step: the largest deviation among
    float64; the tolerance is therefore tied to what such flips do to THIS step: max(2e-3, 5 x the deviation of the oracle
    run in float32, 1.5 x the deviation of the float64 oracle with the masks of its fragile ReLU inputs (|value| < 4e-6,
    found by `_relu_probe`) inverted).  One inverted mask moves the resnet-32 gradient by 9e-4 (2.3e-3 on the worst
    tensor) -- the float64 oracle does that to itself under a one-ulp perturbation of the input."""
    import copy
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    tag, arch, key, B, loss, cls_weight, nesterov = case[:7]
    mode = case[7] if len(case) > 7 else 0
    emb = class_matrix(key) if key else np.eye(64)
    C, D = emb.shape
    om = omodels.build_network(D, arch, input_channels=3, seed=21)
    omodels.randomize(om, seed=22)
    cls = None
    if cls_weight > 0:
        cls = otrain.ClsHead(D, C, seed=23)
        omodels.randomize(cls.params, seed=24)
    graph = utils.build_network(D, arch, input_channels=3)
    eng = Engine(graph, B, emb, loss=loss, cls_weight=cls_weight, num_classes=C, nesterov=nesterov, clipnorm=10.0,
                 mode=mode, use_cuda_graph=tag.startswith('resnet-110-fc'))
    vel = otrain.make_velocity(om, cls if cls_weight > 0 else None)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    g = torch.Generator().manual_seed(31)
    lr = 0.05
    errs = {}
    for step in range(2):
        to_f32_exact(om, cls)
        for v in vel.values():
            v.copy_(v.float().double())
        eng.set_weights(oracle_weights_np(om, cls))
        eng.set_velocity({k: v.numpy() for k, v in vel.items()})
        x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
        y = torch.randint(0, C, (B,), generator=g)
        # noise floor: the same step by the oracle in float32
        om32, cls32 = copy.deepcopy(om), copy.deepcopy(cls)
        otrain.cast_model(om32, torch.float32, cls32)
        vel32 = {k: v.float() for k, v in vel.items()}
        _, grads32, _ = otrain.train_step(om32, x, y, emb_t.float(), vel32, lr, loss, cls32, cls_weight, nesterov, 10.0)
        # ... and the "flip quantum" of THIS step: the float64 oracle re-run with the ReLU masks of its fragile
        # pre-activations (|value| < 4e-6: fp32 accumulation cannot resolve their sign) inverted
        omq, clsq = copy.deepcopy(om), copy.deepcopy(cls)
        velq = {kk: v.clone() for kk, v in vel.items()}
        with _relu_probe() as probe:
            otrain.train_step(omq, x.double(), y, emb_t, velq, lr, loss, clsq, cls_weight, nesterov, 10.0)
        omq, clsq = copy.deepcopy(om), copy.deepcopy(cls)
        velq = {kk: v.clone() for kk, v in vel.items()}
        fragile = probe.fragile()
        gradsq = None
        if fragile:
            with _relu_probe(flip=fragile):
                _, gradsq, _ = otrain.train_step(omq, x.double(), y, emb_t, velq, lr, loss, clsq, cls_weight, nesterov, 10.0)
        obj, grads, norm = otrain.train_step(om, x.double(), y, emb_t, vel, lr, loss, cls, cls_weight, nesterov, 10.0)
        # (global and worst-tensor deviation: the velocity / weight checks below are per tensor)
        floor = max(_grad_errors({k: v.numpy() for k, v in grads32.items()}, grads, norm)[:2])
        quantum = max(_grad_errors({k: v.numpy() for k, v in gradsq.items()}, grads, norm)[:2]) if gradsq is not None else 0.0
        eng.train_step(x, y, lr=lr)
        m = eng.metrics()
        gn, reg = eng.grad_norm_and_reg()
        e = {
            'loss': abs(m['loss'] - float(obj['embed_loss'].detach())) / max(1.0, abs(float(obj['embed_loss'].detach()))),
            'emb': rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].detach().numpy()),
            'acc': abs(m['acc'] - float(obj['acc'].mean())),
            'gnorm': abs(gn - norm) / norm,
            'reg': abs(reg - float(obj['reg'].detach())) / max(float(obj['reg'].detach()), 1e-12),
            'grad_floor_f32_oracle': floor, 'relu_flip_quantum': quantum, 'fragile_relu_inputs': len(fragile),
        }
        if cls_weight > 0:
            e['cls_loss'] = abs(m['cls_loss'] - float(obj['cls_loss'].detach())) / max(1.0, abs(float(obj['cls_loss'].detach())))
        e['grad_global'], e['grad_worst'], worst_name = _grad_errors(eng.get_grads(), grads, norm)
        allp = dict(om.params)
        if cls is not None:
            allp.update(cls.params)
        ew = eng.get_weights()
        e['weights'] = max(rel_l2(ew[n], allp[n].numpy()) for n in allp)
        ev = eng.get_velocity()
        vtot = float(np.sqrt(sum(float(v.norm()) ** 2 for v in vel.values())))
        e['velocity'] = max([rel_l2(ev[n], vel[n].numpy()) for n in vel if float(vel[n].norm()) > 1e-3 * vtot] or [0.0])
        errs[step] = e
        report('train_step', case=tag, mode=mode, step=step, worst_grad_tensor=worst_name, **e)
    for step, e in errs.items():
        gtol = max(2e-3, 5 * e['grad_floor_f32_oracle'], 1.5 * e['relu_flip_quantum'])
        assert e['loss'] < 1e-4 and e['emb'] < 1e-4, (step, e)
        assert e.get('cls_loss', 0.0) < 1e-4, (step, e)
        assert e['gnorm'] < max(1e-4, gtol / 10) and e['reg'] < 1e-5, (step, e)
        assert e['grad_global'] < gtol, (step, e)
        assert e['velocity'] < gtol and e['weights'] < gtol * lr, (step, e)
        assert e['acc'] <= 1.0 / B + 1e-9, (step, e)


def test_inference_uses_moving_statistics():
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import utils
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('cifar100')
    om = omodels.build_network(100, 'resnet-32' if False else 'simple', input_channels=3, seed=5)
    omodels.randomize(om, seed=6)
    to_f32_exact(om)
    graph = utils.build_network(100, 'simple', input_channels=3)
    B = 4
    eng = Engine(graph, B, emb, use_cuda_graph=False)
    eng.set_weights(oracle_weights_np(om))
    g = torch.Generator().manual_seed(1)
    x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
    with torch.no_grad():
        ref = otrain.head_forward(om.forward(x.double(), training=False), 'inv_corr').numpy()
    got = eng.predict(x)
    assert rel_max(got, ref) < 1e-4


def test_fast_mode_error_is_reported_not_hidden():
    """SE_MODE_TF32 (tensor-core inputs with a 10-bit mantissa) is not expected to meet 1e-4; its measured
    deviation from the oracle is recorded so that DESIGN.md can quote it."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import _lib, utils
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('cifar100')
    om = omodels.build_network(100, 'resnet-110-fc', input_channels=3, seed=41)
    to_f32_exact(om)
    graph = utils.build_network(100, 'resnet-110-fc', input_channels=3)
    B = 8
    eng = Engine(graph, B, emb, mode=_lib.SE_MODE_TF32, use_cuda_graph=False)
    eng.set_weights(oracle_weights_np(om))
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
    y = torch.randint(0, 100, (B,), generator=g)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    obj = otrain.train_objective(om, x.double(), y, emb_t)
    eng.load_batch(x, y)
    eng._run('fwdbwd', graph=False)
    e_emb = rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].detach().numpy())
    e_loss = abs(eng.metrics()['loss'] - float(obj['embed_loss']))
    report('fast_mode', emb=e_emb, loss=e_loss)
    assert e_emb < 5e-2 and e_loss < 5e-2


@pytest.mark.parametrize('mode', ['f32', 'tf32x3'])
def test_resnet50_step_matches_oracle(mode):
    """Config 4 architecture (keras.applications ResNet50 v1 + GAP + Dense 'embedding', utils.py:228-243) on a small
    64x64 input: 7x7/2 stem with explicit padding, 3x3/2 max-pool, bottleneck blocks with projection shortcuts, NAB-sized
    (555-d) head.  The backbone itself is third-party and unpinned (DESIGN.md); this checks engine vs oracle."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import _lib
    from semantic_embeddings_b200.models import resnet50
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('nab')
    C, D = emb.shape
    B = 2
    om = omodels.build_resnet50(D, 3, seed=51)
    omodels.randomize(om, seed=52)
    to_f32_exact(om)
    graph = resnet50.ResNet50(D, input_shape=(64, 64, 3))
    # tf32x3: the 1x1 bottleneck convolutions with >= 128 pixels run on the tcgen05 GEMM kernels (conv_tc.cu flat mode,
    # conv1x1_wgrad_tc.cu), the rest on the fp32 kernels
    eng = Engine(graph, B, emb, use_cuda_graph=False, mode=_lib.SE_MODE_TF32X3 if mode == 'tf32x3' else _lib.SE_MODE_F32)
    eng.set_weights(oracle_weights_np(om))
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, 64, 64, 3, generator=g, dtype=torch.float64).float()
    y = torch.randint(0, C, (B,), generator=g)
    vel = otrain.make_velocity(om)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    # noise floor of this ill-conditioned case (batch 2, BatchNorm over 8 values at the 2x2 maps): the same step by the
    # oracle in float32 -- the embedding tolerance is 1e-4 or three times that floor, whichever is larger
    import copy
    om32 = copy.deepcopy(om)
    otrain.cast_model(om32, torch.float32)
    obj32, _, _ = otrain.train_step(om32, x, y, emb_t.float(), {k: v.float() for k, v in vel.items()}, 0.05)
    obj, grads, norm = otrain.train_step(om, x.double(), y, emb_t, vel, 0.05)
    floor = rel_max(obj32['emb'].detach().numpy(), obj['emb'].detach().numpy())
    eng.train_step(x, y, lr=0.05)
    m = eng.metrics()
    e_loss = abs(m['loss'] - float(obj['embed_loss'].detach()))
    e_emb = rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].detach().numpy())
    gg, gw, name = _grad_errors(eng.get_grads(), grads, norm)
    report('resnet50_step_' + mode, loss=e_loss, emb=e_emb, emb_floor_f32_oracle=floor, grad_global=gg, worst=name)
    assert e_loss < 1e-4 and e_emb < max(1e-4, 3 * floor), (e_loss, e_emb, floor)
    # randomly initialised ResNet-50, batch of 2, 2x2 final maps: BN backward is ill-conditioned and a handful of ReLU masks
    # sit within fp32 rounding of zero -- the float32 ORACLE itself deviates from float64 by 1.0e-2 here (1.4e-2 at batch 4 /
    # 96x96, 1.9e-2 at batch 6 / 128x128).  The fp32 kernels measure 1.9e-2, the tensor-core mode (different rounding,
    # different flips) 5.7e-2.
    assert gg < (5e-2 if mode == 'f32' else 1e-1), gg


def test_pairwise_retrieval_api_matches_reference_fixture():
    """The drop-in function (same call as evaluate_retrieval.pairwise_retrieval, evaluate_retrieval.py:22) on the
    dict-of-features form against the rankings the reference's own code produced (make_golden.py)."""
    from semantic_embeddings_b200.evaluate_retrieval import pairwise_retrieval
    d = np.load(os.path.join(G, 'retrieval_ref.npz'))
    fd = {int(i): f.copy() for i, f in zip(d['ids'], d['feat'])}
    r = pairwise_retrieval({'feat': fd}, normalize=False, return_generator=False)
    assert list(r.keys()) == d['rank_dict_keys'].tolist()
    got = np.array(list(r.values()))
    ref = d['rank_dict_vals']
    assert got.shape == ref.shape
    assert (got != ref).mean() < 2e-3          # only fp32-level near-ties may swap
    assert (got[:, 0] == ref[:, 0]).all()       # every query retrieves itself first
    # generator form + normalize=True side effect on a caller-supplied array (evaluate_retrieval.py:58)
    f = d['feat'].copy()
    gen = pairwise_retrieval(f, normalize=True)
    first = next(gen)
    assert first[0] == 0 and first[1][0] == 0
    np.testing.assert_allclose(np.linalg.norm(f, axis=1), 1.0, atol=1e-5)
    with pytest.raises(ValueError):
        pairwise_retrieval({0: np.zeros((2, 3), np.float32), 1: np.zeros((2, 3), np.float32)})


# ----------------------------------------------------------------------------------------------- BASELINE-size parity
# The step tests above use small batches so that the float64 oracle with its ReLU-flip probes stays fast; the cases
# below run the sizes BASELINE.json quotes (many tiles per CTA, full CTA grids, CUDA graph) in the benchmarked
# arithmetic (SE_MODE_TF32X3) against ONE float64 oracle pass each.

def test_resnet110_batch128_step_matches_oracle_in_benchmarked_mode():
    """BASELINE configs[1]: CIFAR-100 ResNet-110(-fc), cosine loss, batch 128, one full training step from a CUDA graph
    in SE_MODE_TF32X3 -- exactly what bench.py times.  Embeddings / loss <= 1e-4, gradient within the fp32 noise floor."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import _lib, utils
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('cifar100')
    B = 128
    om = omodels.build_network(100, 'resnet-110-fc', input_channels=3, seed=61)
    omodels.randomize(om, seed=62)
    to_f32_exact(om)
    eng = Engine(utils.build_network(100, 'resnet-110-fc', input_channels=3), B, emb, mode=_lib.SE_MODE_TF32X3,
                 use_cuda_graph=True)
    eng.set_weights(oracle_weights_np(om))
    g = torch.Generator().manual_seed(63)
    x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
    y = torch.randint(0, 100, (B,), generator=g)
    vel = otrain.make_velocity(om)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    # noise floor of the gradient at this size: the same step by the oracle in float32 (ReLU masks of pre-activations that
    # fp32 cannot resolve flip against float64; the more samples, the more such elements)
    import copy
    om32 = copy.deepcopy(om)
    otrain.cast_model(om32, torch.float32)
    _, grads32, _ = otrain.train_step(om32, x, y, emb_t.float(), {k: v.float() for k, v in vel.items()}, 0.05)
    obj, grads, norm = otrain.train_step(om, x.double(), y, emb_t, vel, 0.05)
    floor = max(_grad_errors({k: v.numpy() for k, v in grads32.items()}, grads, norm)[:2])
    eng.train_step(x, y, lr=0.05)
    m = eng.metrics()
    gn, _ = eng.grad_norm_and_reg()
    e_loss = abs(m['loss'] - float(obj['embed_loss'].detach())) / max(1.0, abs(float(obj['embed_loss'].detach())))
    e_emb = rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].detach().numpy())
    gg, gw, name = _grad_errors(eng.get_grads(), grads, norm)
    ew = eng.get_weights()
    e_w = max(rel_l2(ew[n], om.params[n].numpy()) for n in om.params)
    report('baseline_size', case='resnet-110-fc B=128 step tf32x3 graph', loss=e_loss, emb=e_emb, gnorm=abs(gn - norm) / norm,
           grad_global=gg, grad_worst=gw, worst=name, weights=e_w, grad_floor_f32_oracle=floor)
    assert e_loss < 1e-4 and e_emb < 1e-4, (e_loss, e_emb)
    gtol = max(2e-3, 3 * floor)
    assert abs(gn - norm) / norm < 1e-3 and gg < gtol and e_w < gtol * 0.05, (gn, norm, gg, e_w, floor)


def test_wrn_28_10_batch64_forward_loss_in_benchmarked_mode():
    """BASELINE configs[2] per-GPU shard: WRN-28-10, batch 64, cosine + softmax combined loss (cls_weight 0.1): forward
    pass, both losses and the classifier probabilities in SE_MODE_TF32X3 (160/320/640-channel tensor-core tiles)."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import _lib, utils
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('cifar100')
    B = 64
    om = omodels.build_network(100, 'wrn-28-10', input_channels=3, seed=71)
    omodels.randomize(om, seed=72)
    cls = otrain.ClsHead(100, 100, seed=73)
    omodels.randomize(cls.params, seed=74)
    to_f32_exact(om, cls)
    eng = Engine(utils.build_network(100, 'wrn-28-10', input_channels=3), B, emb, cls_weight=0.1, num_classes=100,
                 mode=_lib.SE_MODE_TF32X3, use_cuda_graph=False)
    eng.set_weights(oracle_weights_np(om, cls))
    g = torch.Generator().manual_seed(75)
    x = torch.randn(B, 32, 32, 3, generator=g, dtype=torch.float64).float()
    y = torch.randint(0, 100, (B,), generator=g)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    with torch.no_grad():
        obj = otrain.train_objective(om, x.double(), y, emb_t, 'inv_corr', cls, 0.1)
    eng.load_batch(x, y)
    eng._run('fwd', graph=False)
    m = eng.metrics()
    e_loss = abs(m['loss'] - float(obj['embed_loss'])) / max(1.0, abs(float(obj['embed_loss'])))
    e_cls = abs(m['cls_loss'] - float(obj['cls_loss'])) / max(1.0, abs(float(obj['cls_loss'])))
    e_emb = rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].numpy())
    report('baseline_size', case='wrn-28-10 B=64 forward tf32x3', loss=e_loss, cls_loss=e_cls, emb=e_emb)
    assert e_loss < 1e-4 and e_cls < 1e-4 and e_emb < 1e-4, (e_loss, e_cls, e_emb)


def test_resnet50_224_forward_matches_oracle():
    """BASELINE configs[3] geometry: ResNet-50 at 224 x 224 x 3 with the 555-d NAB head, batch 4, forward + loss."""
    from oracle import models as omodels
    from oracle import train as otrain
    from semantic_embeddings_b200 import _lib
    from semantic_embeddings_b200.models import resnet50
    from semantic_embeddings_b200.engine import Engine
    emb = class_matrix('nab')
    C, D = emb.shape
    B = 4
    om = omodels.build_resnet50(D, 3, seed=81)
    omodels.randomize(om, seed=82)
    to_f32_exact(om)
    eng = Engine(resnet50.ResNet50(D, input_shape=(224, 224, 3)), B, emb, mode=_lib.SE_MODE_TF32X3, use_cuda_graph=False)
    eng.set_weights(oracle_weights_np(om))
    g = torch.Generator().manual_seed(83)
    x = torch.randn(B, 224, 224, 3, generator=g, dtype=torch.float64).float()
    y = torch.randint(0, C, (B,), generator=g)
    emb_t = torch.as_tensor(emb.astype(np.float32)).double()
    with torch.no_grad():
        obj = otrain.train_objective(om, x.double(), y, emb_t)
    eng.load_batch(x, y)
    eng._run('fwd', graph=False)
    e_loss = abs(eng.metrics()['loss'] - float(obj['embed_loss'])) / max(1.0, abs(float(obj['embed_loss'])))
    e_emb = rel_max(eng.act['head_out'].cpu().numpy(), obj['emb'].numpy())
    report('baseline_size', case='resnet-50 224x224 B=4 forward', loss=e_loss, emb=e_emb)
    assert e_loss < 1e-4 and e_emb < 1e-4, (e_loss, e_emb)


def test_cli_train_feature_dump_then_retrieval_cli(tmp_path, capsys):
    """End to end through the two drop-in scripts (learn_image_embeddings.py:258-275 -> evaluate_retrieval.py:157-208):
    train one epoch on the synthetic dataset with --top_k_acc / --max_decay / --snapshot, write the feature pickle, run
    the retrieval script on it, and check (a) the pickle format, (b) every number of the printed table and the CSV against
    the CPU oracle (oracle/retrieval.py rankings + oracle/hierarchy.py metrics) computed from the SAME pickle."""
    import pickle
    import learn_image_embeddings as lie
    import evaluate_retrieval as er
    from oracle import hierarchy as ohier
    from oracle import retrieval as oret
    emb_p, hier_p = tmp_path / 'emb.pickle', tmp_path / 'hier.txt'
    with open(emb_p, 'wb') as f:
        pickle.dump({'embedding': class_matrix('cifar100'), 'ind2label': list(range(100)),
                     'label2ind': {i: i for i in range(100)}}, f)
    pc = np.load(os.path.join(G, 'cifar_hierarchy.npz'))['parent_child']
    hier_p.write_text('\n'.join('%d %d' % (p, c) for p, c in pc) + '\n')
    feat_p, snap_p, csv_p = tmp_path / 'feat.pickle', tmp_path / 'snap.pickle', tmp_path / 'perf.csv'
    rc = lie.main(['--dataset', 'synthetic:2048', '--data_root', str(tmp_path), '--embedding', str(emb_p), '--architecture',
                   'simple', '--batch_size', '64', '--epochs', '1', '--top_k_acc', '5', '--max_decay', '0.5',
                   '--snapshot', str(snap_p), '--feature_dump', str(feat_p), '--no_progress'])
    assert rc == 0
    log = capsys.readouterr().out
    assert 'Epoch 1/1' in log and 'val_loss' in log and 'val_acc5' in log
    with open(snap_p, 'rb') as f:
        snap = pickle.load(f)
    assert snap['epoch'] == 1 and snap['iterations'] == 32 and len(snap['weights']) > 10 and len(snap['velocity']) > 10
    with open(feat_p, 'rb') as f:
        dump = pickle.load(f)
    feats = dump['feat']
    assert sorted(feats.keys()) == list(range(512)) and feats[0].shape == (100,) and feats[0].dtype == np.float32
    F = np.stack([feats[i] for i in range(512)])
    np.testing.assert_allclose(np.linalg.norm(F, axis=1), 1.0, atol=1e-5)        # l2norm wrapper of --loss inv_corr
    rc = er.main(['--dataset', 'synthetic:2048', '--data_root', str(tmp_path), '--hierarchy', str(hier_p), '--feat', str(feat_p),
                  '--label', 'run', '--plot_max', '20', '--clip_ahp', '30', '--csv', str(csv_p)])
    assert rc == 0
    table = capsys.readouterr().out
    # the oracle on the same pickle
    from semantic_embeddings_b200.datasets import get_data_generator
    y = np.asarray(get_data_generator('synthetic:2048', '', None).labels_test)
    fx = np.load(os.path.join(G, 'retrieval_ref.npz'))
    ranking = oret.rank_stable(oret.pairwise_dist64(F, False))
    ks = list(range(1, 21)) + [50, 100]
    oavg, _ = ohier.hierarchical_precision(ranking, y, fx['wup_lut'], fx['lcs_height_lut'], ks=ks, compute_ahp=30, compute_ap=True)
    row = [ln for ln in table.splitlines() if ln.startswith('run')][0]
    vals = [float(v) for v in row.split('|')[1:]]
    names = ['P@1 (WUP)', 'P@10 (WUP)', 'P@50 (WUP)', 'P@100 (WUP)', 'AHP@30 (WUP)', 'P@1 (LCS_HEIGHT)', 'P@10 (LCS_HEIGHT)',
             'P@50 (LCS_HEIGHT)', 'P@100 (LCS_HEIGHT)', 'AHP@30 (LCS_HEIGHT)', 'AP']
    assert 'AHP@30 (WUP)' in table
    for nm, v in zip(names, vals):
        assert abs(v - oavg[nm]) < 2e-4, (nm, v, oavg[nm])           # the table prints 4 decimals
    lines = csv_p.read_text().strip().splitlines()
    assert lines[0] == 'k;run' and len(lines) == 21
    for k in range(1, 21):
        kk, v = lines[k].split(';')
        assert int(kk) == k and abs(float(v) - oavg['P@%d (LCS_HEIGHT)' % k]) < 2e-4


def test_cli_finetune_from_dump(tmp_path, capsys):
    """--finetune / --finetune_init through the CLI (learn_image_embeddings.py:183-207): weights are loaded by name from a
    dump of a DIFFERENT head size (the 100-d 'embedding' layer of the dump does not fit the 64-d one of this run and is
    skipped, like Keras' skip_mismatch), the new layers train alone for one epoch -- the backbone in the written snapshot
    is then still the dump's -- and the full model trains afterwards."""
    import pickle
    import learn_image_embeddings as lie
    emb100, emb64 = tmp_path / 'emb100.pickle', tmp_path / 'emb64.pickle'
    rng = np.random.RandomState(3)
    E64 = rng.randn(100, 64)
    E64 /= np.linalg.norm(E64, axis=1, keepdims=True)
    for pth, E in ((emb100, class_matrix('cifar100')), (emb64, E64)):
        with open(pth, 'wb') as f:
            pickle.dump({'embedding': E, 'ind2label': list(range(100)), 'label2ind': {i: i for i in range(100)}}, f)
    dump_p, snap_p = tmp_path / 'pre.pickle', tmp_path / 'snap.pickle'
    common = ['--dataset', 'synthetic:1024', '--data_root', str(tmp_path), '--architecture', 'simple', '--batch_size', '64',
              '--no_progress']
    assert lie.main(common + ['--embedding', str(emb100), '--epochs', '1', '--model_dump', str(dump_p)]) == 0
    capsys.readouterr()
    with open(dump_p, 'rb') as f:
        pre = pickle.load(f)['weights']
    # phase 1 only (--epochs 0 is not expressible: the schedule decides; stop after the frozen phase by looking at the log
    # of a run whose full-model phase is one short epoch)
    assert lie.main(common + ['--embedding', str(emb64), '--epochs', '1', '--finetune', str(dump_p), '--finetune_init', '1',
                              '--snapshot', str(snap_p)]) == 0
    log = capsys.readouterr().out
    assert 'Loading pre-trained weights' in log and 'Pre-training new layers' in log and 'Full model training' in log
    skipped = [ln for ln in log.splitlines() if 'tensors loaded' in ln][0]
    assert ' 2 skipped' in skipped, skipped                  # embedding/kernel and embedding/bias: 100-d dump vs 64-d model
    with open(snap_p, 'rb') as f:
        snap = pickle.load(f)
    assert snap['weights']['embedding/kernel'].shape[1] == 64
    # after the full-model epoch every backbone tensor has moved away from the dump
    name = [n for n in pre if n.endswith('/kernel') and n != 'embedding/kernel'][0]
    assert pre[name].shape == snap['weights'][name].shape and not np.array_equal(pre[name], snap['weights'][name])


def test_bench_dump_outputs_are_the_last_timed_step_and_reproducible(tmp_path):
    """bench.py --dump-outputs: the last timed training step's per-sample loss / accuracy, embeddings, gradient norm and
    updated weights / momentum as float32 / float64 .npy files.  That step starts from the seeded initial state, so two
    runs whose last step trains on the same batch of the 4-batch pool (--steps 2 and --steps 6) write the same numbers up
    to the ordering of atomically accumulated sums (measured on the B200: ~1e-7 in the forward pass, up to 3e-3 of the
    largest momentum value)."""
    import subprocess
    import sys
    from semantic_embeddings_b200 import utils
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for steps in (2, 6):
        d = tmp_path / ('steps%d' % steps)
        out = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--steps', str(steps), '--warmup', '3',
                              '--skip-retrieval', '--skip-cpu-baseline', '--dump-outputs', str(d)],
                             capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])['steps'] == steps
        dumps.append({f[:-4]: np.load(str(d / f)) for f in sorted(os.listdir(str(d)))})
    a, b = dumps
    assert sorted(a) == ['acc', 'embeddings', 'grad_norm_and_l2', 'loss', 'velocity', 'weights']
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a['loss'].shape == (128,) and a['embeddings'].shape == (128, 100) and a['grad_norm_and_l2'].dtype == np.float64
    np.testing.assert_allclose(np.linalg.norm(a['embeddings'], axis=1), 1.0, atol=1e-5)
    g = utils.build_network(100, 'resnet-110-fc', input_channels=3)
    assert a['weights'].size == sum(int(np.prod(p.shape)) for p in g.params.values())
    assert np.isfinite(a['weights']).all() and np.abs(a['velocity']).max() > 0
    tol = {'velocity': 3e-2, 'grad_norm_and_l2': 1e-3}
    for k in a:
        err = rel_max(b[k], a[k])
        report('bench_dump_outputs', array=k, rel_max_err=err)
        assert err <= tol.get(k, 1e-4), (k, err)
