"""The cropped-object support inputs (metain_type 3 / 4, and the plain image of type 1) on the GPU: the <= 8-channel
first-layer kernels, the engine's routing to them, the mini model against the reference (tests/golden/metain.npz) and
the float64 oracle, the graphed step, the input pipeline, the ensemble and the weight file."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
CHANNELS = {1: 3, 2: 4, 3: 7, 4: 6}
TOL = 1e-3


def rel(a, b):
    a = np.asarray(a.detach().double().cpu() if torch.is_tensor(a) else a, np.float64)
    b = np.asarray(b.detach().double().cpu() if torch.is_tensor(b) else b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


def st():
    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope='module')
def gold():
    return np.load(os.path.join(G, 'metain.npz'), allow_pickle=False)


@pytest.fixture()
def metain():
    """cfg.metain_type for the test, restored afterwards."""
    from fewshot_detection_b200.cfg import cfg
    old = cfg.metain_type
    yield cfg
    cfg.metain_type = old


@pytest.fixture(params=['fp32', 'tc'])
def path(request):
    from fewshot_detection_b200 import engine
    old = engine.USE_TC
    engine.USE_TC = request.param == 'tc'
    yield request.param
    engine.USE_TC = old


# ------------------------------------------------------------------------------------------------ first-layer kernels
@pytest.mark.parametrize('C', [5, 6, 7, 8])
@pytest.mark.parametrize('B,H,W,Cout', [(2, 13, 17, 32), (3, 64, 64, 16), (1, 5, 3, 8), (2, 416, 416, 32), (5, 200, 130, 32),
                                        (7, 100, 211, 24), (1, 40, 512, 32)])
def test_first_layer_8ch_fwd_stats_wgrad(B, H, W, Cout, C):
    from fewshot_detection_b200 import _lib as L
    C0, C1 = (6, C - 6) if C >= 6 else (3, C - 3)          # image + crop [+ mask], or a 3 + 2 split
    g = torch.Generator(device='cuda').manual_seed(H + W + C)
    a = torch.rand(B, C0, H, W, device='cuda', generator=g)
    m = torch.rand(B, C1, H, W, device='cuda', generator=g) if C1 else None
    x = torch.cat([a, m], 1) if C1 else a
    w = (torch.randn(Cout, C, 3, 3, device='cuda', generator=g) * 0.2).double().requires_grad_(True)
    dz = torch.randn(B, Cout, H, W, device='cuda', generator=g)
    ref = F.conv2d(x.double(), w, None, 1, 1)
    ref.backward(dz.double())
    wp = torch.zeros(Cout, 9, 8, device='cuda')                # channel pitch 8 above 4 channels
    wp[:, :, :C] = w.detach().float().permute(0, 2, 3, 1).reshape(Cout, 9, C)
    z = torch.empty(B * H * W, Cout, device='cuda')
    L.call('fsdet_conv_first_fwd', a.data_ptr(), C0, m.data_ptr() if C1 else None, C1, wp.data_ptr(), z.data_ptr(), Cout, B, H, W,
           Cout, st())
    assert rel(z.view(B, H, W, Cout).permute(0, 3, 1, 2), ref) < 1e-5
    z2 = torch.empty(B * H * W, Cout + 4, device='cuda')
    rows = L.lib.fsdet_conv_first_stat_rows(B, H, W)
    part = torch.full((rows, 4 * Cout), 123.0, device='cuda')
    L.call('fsdet_conv_first_fwd_stats', a.data_ptr(), C0, m.data_ptr() if C1 else None, C1, wp.data_ptr(), z2.data_ptr(), Cout + 4,
           B, H, W, Cout, part.data_ptr(), st())
    assert torch.equal(z2[:, :Cout], z)
    sp = part.double().sum(0)
    assert rel(sp[:Cout], z.double().sum(0)) < 1e-5 or (sp[:Cout] - z.double().sum(0)).abs().max() < 1e-3
    assert rel(sp[Cout:2 * Cout], (z.double() ** 2).sum(0)) < 1e-5
    assert torch.equal(part[:, 2 * Cout:3 * Cout].min(0)[0], z.min(0)[0])
    assert torch.equal(part[:, 3 * Cout:].max(0)[0], z.max(0)[0])
    assert L.lib.fsdet_conv_first_wgrad_supported(C, W)
    dzb = dz.permute(0, 2, 3, 1).contiguous().view(-1, Cout)
    nws = L.lib.fsdet_conv_first_wgrad_workspace_floats_cin(B, H, W, C, Cout)
    ws = torch.empty(nws, device='cuda')
    dw = torch.full((Cout, 9, 8), 7.0, device='cuda')
    L.call('fsdet_conv_first_wgrad', a.data_ptr(), C0, m.data_ptr() if C1 else None, C1, dzb.data_ptr(), Cout, dw.data_ptr(),
           ws.data_ptr(), nws, B, H, W, Cout, st())
    assert rel(dw.view(Cout, 3, 3, 8)[:, :, :, :C].permute(0, 3, 1, 2), w.grad) < 1e-5
    assert (dw[:, :, C:] == 0).all()


def test_first_layer_wgrad_support_limit():
    """The 8-channel weight gradient stages its rows in shared memory up to W = 518; past it the call is refused
    (the engine takes the NHWC path there, see test_support_net_routes_by_width)."""
    from fewshot_detection_b200 import _lib as L
    assert L.lib.fsdet_conv_first_wgrad_supported(7, 512) and not L.lib.fsdet_conv_first_wgrad_supported(7, 544)
    assert L.lib.fsdet_conv_first_wgrad_supported(4, 608) and not L.lib.fsdet_conv_first_wgrad_supported(9, 64)
    B, H, W, Cout = 1, 4, 608, 32
    a = torch.rand(B, 7, H, W, device='cuda')
    dz = torch.randn(B * H * W, Cout, device='cuda')
    nws = L.lib.fsdet_conv_first_wgrad_workspace_floats_cin(B, H, W, 7, Cout)
    ws = torch.empty(nws, device='cuda')
    dw = torch.empty(Cout, 9, 8, device='cuda')
    with pytest.raises(RuntimeError):
        L.call('fsdet_conv_first_wgrad', a.data_ptr(), 7, None, 0, dz.data_ptr(), Cout, dw.data_ptr(), ws.data_ptr(), nws, B, H, W,
               Cout, st())


# ------------------------------------------------------------------------------------------------ models
def _meta(t, seed, c=4, out=128, side=128, meta_side=64):
    from fewshot_detection_b200.darknet_meta import Darknet
    from fewshot_detection_b200 import netcfg
    from seeding import seeded_init
    det = netcfg.mini_dynamic_blocks(side, c)
    ler = netcfg.mini_reweighting_blocks(meta_side, c, out, channels=CHANNELS[t])
    m = Darknet([dict(b) for b in det], [dict(b) for b in ler])
    seeded_init(m, seed)
    return m.cuda().train()


@pytest.mark.parametrize('t', [3, 4])
@pytest.mark.parametrize('W', [64, 576])
def test_support_net_routes_by_width(metain, t, W):
    """The support net's first convolution reads the 6- or 7-channel NCHW input through first_fwd / first_wgrad where
    the weight-gradient staging fits, and the generic NHWC kernels past it - with the same result."""
    from seeding import synth_masks
    metain.metain_type = t
    m = _meta(t, 5, meta_side=W)
    metax = torch.rand(2, 6, W, W, device='cuda')
    mask = torch.from_numpy(synth_masks(2, W, 3)).cuda()
    m._ler.profile = {}
    dw = m.meta_forward(metax, mask)[0]
    dw.sum().backward()
    names = set(k for k in m._ler.profile if not k.startswith('_'))
    m._ler.profile = None
    direct = m.learnet_models[0][0].weight.grad.detach().clone()
    if W <= 518:
        assert 'first_fwd' in names and 'first_wgrad' in names, names
    else:
        assert 'first_fwd' not in names and 'first_wgrad' not in names, names
    # float64 CPU oracle of the same support net
    from test_metain_host_emul import oracle_meta
    from fewshot_detection_b200 import netcfg
    from seeding import seeded_init
    om = oracle_meta(netcfg.mini_dynamic_blocks(128, 4), netcfg.mini_reweighting_blocks(W, 4, 128, channels=CHANNELS[t]), t)
    seeded_init(om, 5)
    om.double().train()
    odw = om.meta_forward(metax.double().cpu(), mask.double().cpu())[0]
    odw.sum().backward()
    assert rel(dw, odw) < 1e-4
    assert rel(direct, om.learnet_models[0][0].weight.grad) < 1e-3


@pytest.mark.parametrize('t', [1, 3, 4])
def test_meta_mini_vs_reference(gold, metain, path, t):
    metain.metain_type = t
    bs, cs, side, ms, seed, seen = (int(v) for v in gold['model/dims'])
    key = 'model/in%d/' % t
    from test_metain_host_emul import regen_inputs
    m = _meta(t, seed)
    x, metax, mask, target = regen_inputs(gold, t)
    x, metax, mask = x.cuda(), metax.cuda(), mask.cuda()
    m._ler.profile = {}
    out = m(x, metax, mask)
    if t != 1:
        assert 'first_fwd' in m._ler.profile
    m._ler.profile = None
    assert rel(out, gold[key + 'output']) < TOL
    L = m.models[len(m.models) - 1]
    L.seen = seen
    loss = L(out, target)
    loss.backward()
    assert abs(loss.item() - float(gold[key + 'loss'])) < TOL * abs(float(gold[key + 'loss']))
    for name, p in m.named_parameters():
        g = p.grad.detach().cpu().contiguous()
        if key + 'grad/' + name in gold.files:
            assert rel(g, gold[key + 'grad/' + name]) < TOL, name
        else:
            gn = float(gold[key + 'gradnorm/' + name])
            assert abs(g.double().norm().item() - gn) < TOL * gn + 1e-12, name
            assert rel(g.reshape(-1)[:64], gold[key + 'gradhead/' + name]) < 1e-2, name


@pytest.mark.parametrize('t', [1, 3, 4])
def test_meta_mini_vs_float64_oracle(metain, t):
    """Support-net gradients against the float64 oracle on fresh seeded inputs; like the existing full-model check,
    the bar is max(1e-3, 3 x the float32 oracle's distance), and it must hold for the median of three batch seeds."""
    from oracle import region_loss as ORL
    from test_metain_host_emul import oracle_meta
    from fewshot_detection_b200 import netcfg
    from seeding import seeded_init, synth_masks, synth_targets
    metain.metain_type = t
    det, ler = netcfg.mini_dynamic_blocks(128, 4), netcfg.mini_reweighting_blocks(64, 4, 128, channels=CHANNELS[t])
    worst = []
    for s in (1, 2, 3):
        g = torch.Generator().manual_seed(900 + s)
        x = torch.rand(2, 3, 128, 128, generator=g)
        metax = torch.rand(3, 3 if t == 1 else 6, 64, 64, generator=g)
        mask = torch.from_numpy(synth_masks(3, 64, 910 + s))
        tgt = torch.from_numpy(synth_targets(2, 3, 920 + s, max_gt=4))
        grads = {}
        for dt in (torch.float64, torch.float32):
            om = oracle_meta([dict(b) for b in det], [dict(b) for b in ler], t)
            seeded_init(om, 51)
            om = om.to(dt).train()
            oo = om(x.to(dt), metax.to(dt), mask.to(dt))
            o32 = oo.detach().float().requires_grad_(True)
            ORL.region_loss_v2(o32, tgt, om.anchors, om.num_anchors, om.num_classes, seen=20000).backward()
            oo.backward(o32.grad.to(dt))
            grads[dt] = {n: p.grad.detach().double() for n, p in om.named_parameters()}
        m = _meta(t, 51)
        Lr = m.models[len(m.models) - 1]
        Lr.seen = 20000
        Lr(m(x.cuda(), metax.cuda(), mask.cuda()), tgt).backward()
        w = 0.0
        for n, p in m.named_parameters():
            if not n.startswith('learnet_models'):
                continue
            e_ref = rel(grads[torch.float32][n], grads[torch.float64][n])
            e = rel(p.grad, grads[torch.float64][n])
            w = max(w, e / max(TOL, 3 * e_ref))
        worst.append(w)
    assert sorted(worst)[1] < 1.0, worst


def test_graphed_step_matches_eager_type3(metain):
    from fewshot_detection_b200.optim import FusedSGD
    from fewshot_detection_b200.distributed import GradAllReducer
    from fewshot_detection_b200.graph import GraphedTrainStep
    from seeding import synth_targets, synth_masks
    metain.metain_type = 3
    bs, cs = 4, 3

    def batch(it):
        g = torch.Generator().manual_seed(100 + it)
        x = torch.rand(bs, 3, 128, 128, generator=g).cuda()
        metax = torch.rand(cs, 6, 64, 64, generator=g).cuda()
        return x, metax, torch.from_numpy(synth_masks(cs, 64, 200 + it)).cuda(), torch.from_numpy(synth_targets(bs, cs, 300 + it, max_gt=4))

    runs = []
    for graph in (False, True):
        m = _meta(3, 11, c=8, out=256)
        opt = FusedSGD(m.parameters(), lr=1e-3, momentum=0.9, dampening=0, weight_decay=5e-4)
        L = m.models[len(m.models) - 1]
        L.verbose = False
        L.seen = 20000
        red = GradAllReducer(m)
        gs = GraphedTrainStep(m, L, opt, red) if graph else None
        losses = []
        for it in range(4):
            x, metax, mask, tgt = batch(it)
            L.seen += bs
            if graph:
                losses.append(gs(x, metax, mask, tgt).item())
            else:
                red.begin_step()
                loss = L(m(x, metax, mask), tgt)
                loss.backward()
                red.finish()
                opt.step()
                losses.append(loss.item())
        runs.append((losses, [p.detach().clone() for p in m.parameters()]))
    (l0, p0), (l1, p1) = runs
    for a, b in zip(l0, l1):
        assert abs(a - b) <= 1e-5 * abs(a), (l0, l1)
    for a, b in zip(p0, p1):
        assert rel(b, a) < 1e-5


# ------------------------------------------------------------------------------------------------ input pipeline
@pytest.fixture()
def cfg48(metain):
    cfg = metain
    keys = ('data', 'multiscale', 'metayolo', 'yolo_joint', 'classes', 'base_classes', 'base_ids', 'meta_width', 'meta_height',
            'mask_width', 'mask_height')
    old = {k: cfg.get(k) for k in keys}
    cfg.data, cfg.multiscale, cfg.metayolo, cfg.yolo_joint = 'voc', 0, True, False
    cfg.classes = cfg.voc_classes
    cfg.base_classes, cfg.base_ids = cfg.voc_classes[:3], list(range(3))
    cfg.meta_width = cfg.meta_height = cfg.mask_width = cfg.mask_height = 48
    yield cfg
    for k, v in old.items():
        if v is None:
            cfg.pop(k, None)
        else:
            cfg[k] = v


@pytest.mark.parametrize('t', [3, 4])
@pytest.mark.parametrize('mode', ['train', 'ensemble'])
def test_meta_batcher_on_gpu_equals_reference(gold, cfg48, t, mode):
    from test_metain_host_emul import run_batcher
    metax, mask, ids, key = run_batcher(gold, cfg48, t, mode)
    assert np.array_equal(mask, gold[key + 'mask_u8'].astype(np.float32))
    assert np.array_equal(metax, gold[key + 'img_u8'].astype(np.float32) / np.float32(255))


def test_ensemble_dynamic_weights_type3(gold, cfg48):
    """valid.ensemble_dynamic_weights over type-3 support batches (6 image channels + mask) equals the mean of the
    per-image reweighting vectors of each class."""
    from test_metain_host_emul import _batcher
    from fewshot_detection_b200.valid import ensemble_dynamic_weights
    mb, inds, key = _batcher(gold, cfg48, 3, 'ensemble')
    m = _meta(3, 7, meta_side=48)
    m.eval()
    batches = [mb.batch(range(b, min(b + 3, len(inds)))) for b in range(0, len(inds), 3)]
    ens = ensemble_dynamic_weights(m, batches, 3)
    with torch.no_grad():
        per = torch.cat([m.meta_forward(x, k)[0] for x, k, _ in batches])
    ids = torch.tensor(sum([c for _, _, c in batches], []))
    want = torch.stack([per[ids.cuda() == c].mean(0) for c in range(3)])
    assert rel(ens[0].reshape(want.shape), want) < 1e-5


def test_weight_file_roundtrip_type3(metain, tmp_path):
    metain.metain_type = 3
    m = _meta(3, 21)
    m.seen = 99
    f = str(tmp_path / 'in3.weights')
    m.save_weights(f)
    m2 = _meta(3, 22)
    m2.load_weights(f)
    assert m2.seen == 99
    for (n1, p), (_, q) in zip(m.named_parameters(), m2.named_parameters()):
        assert torch.equal(p.detach().cpu(), q.detach().cpu()), n1
    assert m2.learnet_models[0][0].weight.shape[1] == 7
