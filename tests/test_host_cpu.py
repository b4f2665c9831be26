"""CPU-side checks: the C-ABI library loads and exports exactly what include/c2m_sm100.h
declares, the drop-in boundaries keep the reference's names / signatures / error behaviour,
the registry + yaml API resolve, and state-dict keys match the reference nets (strict load)."""
import copy
import inspect
import os
import re
import subprocess

import pytest
import torch

import seeding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def built():
    import __graft_entry__ as g
    g.build()
    from c2m_b200 import _lib
    return _lib


def _header_functions():
    src = open(os.path.join(ROOT, 'include', 'c2m_sm100.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(c2m_[a-z0-9_]+)\s*\(', src)))


def test_library_exports_every_declared_symbol(built):
    declared = _header_functions()
    assert 'c2m_corr_argmax_f32' in declared and 'c2m_dcn_v2_forward_f32' in declared
    out = subprocess.run(['nm', '-D', '--defined-only', built.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r'\bT (c2m_[a-z0-9_]+)', out))
    assert set(declared) <= exported, set(declared) - exported
    assert set(built.SYMBOLS) == set(declared)          # the ctypes table binds all of them
    lib = built.lib()
    assert lib.c2m_abi_version() == 4


def test_sass_is_blackwell_native(built):
    sass = subprocess.run(['cuobjdump', '-sass', built.LIB_PATH], capture_output=True, text=True).stdout
    if not sass:
        pytest.skip('cuobjdump not available')
    assert 'UTCHMMA' in sass and 'UTMALDG' in sass and 'LDTM' in sass   # tcgen05.mma / TMA / tcgen05.ld
    assert 'sm_100a' in sass or 'SM100a' in sass.replace('sm_100', 'SM100')


def test_workspace_query_and_error_string(built):
    lib = built.lib()
    n = lib.c2m_corr_workspace_bytes(1, 256, 40, 40, 125, 125, 3, 1, 1)
    assert n > 4 * 256 * (40 * 40 + 125 * 125)
    assert lib.c2m_corr_workspace_bytes(1, 256, 2, 40, 125, 125, 3, 1, 1) == 0
    assert b'smaller than the patch' in lib.c2m_last_error()


def test_ext_module_surface():
    import _ext
    for name in ('dcn_v2_forward', 'dcn_v2_backward', 'dcn_v2_psroi_pooling_forward', 'dcn_v2_psroi_pooling_backward'):
        assert callable(getattr(_ext, name))       # DCNv2/src/vision.cpp:3-8
    params = list(inspect.signature(_ext.dcn_v2_forward).parameters)
    assert params == ['input', 'weight', 'bias', 'offset', 'mask', 'kernel_h', 'kernel_w', 'stride_h', 'stride_w',
                      'pad_h', 'pad_w', 'dilation_h', 'dilation_w', 'deformable_group']   # dcn_v2.h:9-22


def test_cpu_tensors_fail_loudly():
    """No CPU fallback: reference `_ext` raises 'Not implemented on the CPU' (dcn_v2.h:38)."""
    import _ext
    from mmsr.models.archs.ref_map_util import feature_match_index
    x = torch.zeros(1, 8, 6, 6)
    with pytest.raises(RuntimeError, match='CUDA tensor'):
        _ext.dcn_v2_forward(x, torch.zeros(8, 8, 3, 3), torch.zeros(8), torch.zeros(1, 18, 6, 6),
                            torch.zeros(1, 9, 6, 6), 3, 3, 1, 1, 1, 1, 1, 1, 1)
    with pytest.raises(RuntimeError, match='CUDA tensor'):
        feature_match_index(torch.zeros(8, 6, 6), torch.zeros(8, 6, 6))
    with pytest.raises((RuntimeError, TypeError)):
        _ext.dcn_v2_backward(*([x] * 6), 3, 3, 1, 1, 1, 1, 1, 1, 1)


def test_feature_match_index_signature():
    from mmsr.models.archs.ref_map_util import feature_match_index, sample_patches
    sig = inspect.signature(feature_match_index)
    assert list(sig.parameters) == ['feat_input', 'feat_ref', 'patch_size', 'input_stride', 'ref_stride', 'is_norm',
                                    'norm_input']                       # ref_map_util.py:26-32
    d = {k: v.default for k, v in sig.parameters.items() if v.default is not inspect._empty}
    assert d == dict(patch_size=3, input_stride=1, ref_stride=1, is_norm=True, norm_input=False)
    p = sample_patches(torch.arange(2 * 4 * 5.).view(2, 4, 5))
    assert p.shape == (2, 3, 3, 6) and p[1, 2, 1, 4].item() == 20 + (1 + 2) * 5 + (1 + 1)


def test_state_dict_keys_match_reference_nets():
    from mmsr.models.archs.contras_extractor_arch import ContrasExtractorSep
    from mmsr.models.archs.corres_generation_arch import CorrespondenceGenerationArch
    from mmsr.models.archs.ref_restoration_arch import RestorationNet
    for net, spec in ((RestorationNet(64, 16, 8), seeding.spec_restoration_net()),
                      (ContrasExtractorSep(), seeding.spec_extractor()),
                      (CorrespondenceGenerationArch(), seeding.spec_net_map())):
        sd = net.state_dict()
        assert {k: tuple(v.shape) for k, v in sd.items()} == {k: tuple(v) for k, v in spec.items()}
        net.load_state_dict(seeding.seeded_state_dict(spec, 3), strict=True)
    g = RestorationNet()
    for size in ('small', 'medium', 'large'):       # conv_offset_mask is zero-initialised (ref_restoration_arch.py:42-49)
        m = getattr(g.dyn_agg_restore, f'{size}_dyn_agg').conv_offset_mask
        assert m.weight.abs().sum() == 0 and m.bias.abs().sum() == 0
    # a DataParallel-style checkpoint (module. prefix) is accepted by the model wrapper's loader
    from mmsr.models.ref_restoration_model import RefRestorationModel
    assert hasattr(RefRestorationModel, 'load_network') and hasattr(RefRestorationModel, 'validation')


def test_yaml_registry_roundtrip():
    from mmsr.models import networks
    from mmsr.models.archs import _arch_modules
    from mmsr.utils.options import dict2str, dict_to_nonedict, parse
    opt = dict_to_nonedict(parse(os.path.join(ROOT, 'tests', 'fixtures', 'test_c2m_synth.yml'), is_train=False))
    assert opt['crop_border'] == 4 and opt['is_train'] is False and opt['no_such_key'] is None
    assert opt['datasets']['test_1']['phase'] == 'test' and opt['datasets']['test_1']['scale'] == 4
    assert opt['path']['visualization'].endswith(os.path.join('results', 'c2m_synth', 'visualization'))
    assert 'network_g' in dict2str(opt)
    names = {m.__name__.rsplit('.', 1)[1] for m in _arch_modules}
    assert {'ref_restoration_arch', 'corres_generation_arch', 'contras_extractor_arch'} <= names
    o = copy.deepcopy(opt)
    assert type(networks.define_net_g(o)).__name__ == 'RestorationNet'
    assert type(networks.define_net_map(o)).__name__ == 'CorrespondenceGenerationArch'
    assert type(networks.define_net_extractor(o)).__name__ == 'ContrasExtractorSep'
    with pytest.raises(ValueError):
        networks.dynamical_instantiation(_arch_modules, 'NoSuchArch', {})


def test_model_wrapper_needs_cuda():
    from mmsr.models import create_model
    from mmsr.utils.options import dict_to_nonedict, parse
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    opt = dict_to_nonedict(parse(os.path.join(ROOT, 'tests', 'fixtures', 'test_c2m_synth.yml'), is_train=False))
    with pytest.raises(RuntimeError, match='CUDA'):
        create_model(opt)


def test_dataset_sample_dict():
    from mmsr.data import create_dataloader, create_dataset
    ds = create_dataset({'type': 'SyntheticRefDataset', 'name': 's', 'num': 2, 'gt_size': 64, 'ref_size': 40, 'scale': 4,
                         'phase': 'test'})
    s = next(iter(create_dataloader(ds, {'phase': 'test', 'num_workers': 0})))
    assert tuple(s['img_in_lq'].shape) == (1, 3, 16, 16) and tuple(s['img_ref'].shape) == (1, 3, 64, 64)
    assert s['img_ref'][0, :, 40:, :].abs().sum() == 0 and s['img_ref'][0, :, :, 40:].abs().sum() == 0   # zero pad
    # batches keep non-tensor fields as per-sample lists (collate_pairs), so ragged batches of B > 1 pairs work
    assert s['padding'] == [True] and [tuple(int(v) for v in o) for o in s['original_size']] == [(64, 64)]


def test_metrics_and_tensor2img():
    import numpy as np
    from mmsr.utils import metrics
    from mmsr.utils.util import tensor2img
    t = torch.tensor([[[0.0, 1.0]], [[0.5, 0.25]], [[1.0, 2.0]]])           # RGB CHW, one value > 1
    img = tensor2img(t)
    assert img.shape == (1, 2, 3) and img[0, 0].tolist() == [255.0, 128.0, 0.0] and img[0, 1, 0] == 255.0
    a = np.zeros((16, 16, 3)); b = a.copy(); b[8, 8, 0] = 16
    assert abs(metrics.psnr(a, b, crop_border=4) - 20 * np.log10(255 / np.sqrt(256 / (8 * 8 * 3)))) < 1e-9
    assert metrics.psnr(a, a) == float('inf')
    y = metrics.bgr2ycbcr(np.ones((2, 2, 3), np.float32), only_y=True)
    assert abs(float(y[0, 0]) - 235.0 / 255.0) < 1e-6
    assert 0.99 < metrics.ssim(np.random.default_rng(0).random((32, 32)) * 255, np.random.default_rng(0).random((32, 32)) * 255) <= 1.0


def test_specs_equal_real_reference_classes():
    """The hand-written key/shape specs == the state dicts of the reference constructors (fixture:
    reference_specs.json, minted from the reference classes by make_golden.py)."""
    import json
    with open(os.path.join(ROOT, 'tests', 'golden', 'reference_specs.json')) as f:
        got = json.load(f)
    for n, spec in (('g', seeding.spec_restoration_net()), ('e', seeding.spec_extractor()), ('m', seeding.spec_net_map())):
        assert got[n] == {k: list(v) for k, v in spec.items()}


def test_dataset_matches_reference_dataset_golden(tmp_path):
    """N2: the test-phase RefCUFEDDataset (mod-crop, zero-pad to a common size, PIL bicubic /4 and x4,
    BGR->RGB CHW) reproduces the reference class's samples bit-for-bit (fixture: dataset.npz, minted
    from mmsr/data/ref_cufed_dataset.py on the same PNGs)."""
    import numpy as np
    import make_golden as mg
    from mmsr.data import create_dataset
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'dataset.npz'))
    ann = mg.dataset_pngs(str(tmp_path))
    ds = create_dataset({'type': 'RefCUFEDDataset', 'name': 'g', 'dataroot_in': str(tmp_path), 'dataroot_ref': str(tmp_path),
                         'ann_file': ann, 'io_backend': {'type': 'disk'}, 'scale': 4, 'phase': 'test'})
    assert len(ds) == 2
    for i in range(2):
        s = ds[i]
        for k in ('img_in', 'img_in_lq', 'img_in_up', 'img_ref', 'img_ref_lq', 'img_ref_up'):
            assert np.array_equal(s[k].numpy(), g[f'{i}/{k}']), (i, k)
        assert bool(s['padding']) == bool(g[f'{i}/padding'])
        assert list(s['original_size']) == list(g[f'{i}/original_size'])


def test_lazy_result_dicts_behave_like_the_reference_dicts(monkeypatch):
    """`pre_offset` / `img_ref_feat` of CorrespondenceGenerationArch.forward are plain dicts in the
    reference (corres_generation_arch.py:107-116); here they fill themselves on first access.
    Host logic only: the device conversions are replaced by CPU stand-ins."""
    import torch
    from c2m_b200 import ops
    from mmsr.models.archs import corres_generation_arch as cg
    from mmsr.models.archs import vgg_arch

    calls = []

    def fake_to_f32(p, add=None, channels_last=False):
        calls.append(p)
        return torch.full((1, 2, 3, 3), float(p))

    monkeypatch.setattr(ops, 'psa_to_f32', fake_to_f32)
    feats = vgg_arch.PackedFeatures({'relu1_1': 1, 'relu2_1': 2})
    assert len(feats) == 2 and 'relu1_1' in feats and 'relu3_1' not in feats and not calls
    assert feats.psa('relu2_1') == 2 and not calls
    assert float(feats['relu2_1'].mean()) == 2.0 and calls == [2]
    assert feats['relu2_1'] is feats['relu2_1'] and calls == [2]           # cached
    assert feats.get('relu3_1') is None and feats.get('relu1_1').shape == (1, 2, 3, 3)
    assert sorted(feats.keys()) == ['relu1_1', 'relu2_1'] and len(list(feats.items())) == 2
    try:
        feats['relu9_9']
        raise AssertionError('missing layer must raise KeyError')
    except KeyError:
        pass

    built = []

    def fake_pyramid(idx, scale, ref_gw=None):
        built.append(scale)
        return torch.zeros(1, 9, 4 * scale, 4 * scale, 2)

    monkeypatch.setattr(cg._ops, 'offset_pyramid', fake_pyramid)
    pre = cg.PreOffsets(torch.zeros(1, 2, 2, dtype=torch.int64), 2)
    assert len(pre) == 3 and 'relu2_1' in pre and not built
    h = pre.handle('relu1_1')
    assert (h.scale, h.ref_gw) == (4, 2) and not built
    assert pre['relu2_1'].shape == (1, 9, 8, 8, 2) and built == [2]
    assert pre.get('nope', 7) == 7 and set(pre.keys()) == {'relu1_1', 'relu2_1', 'relu3_1'}
    assert sorted(built) == [1, 2, 4]


def test_net_map_vgg_defaults_to_imagenet_weights(tmp_path, monkeypatch):
    """ADVICE r1 (high): the reference builds net_map's VGG19 with `pretrained=True` and never loads it from a
    checkpoint (vgg_arch.py:103-104), so the reference YAML (no extra key) must yield ImageNet weights here too —
    from a local torchvision checkpoint — and must RAISE when there are none, not run on random weights."""
    import torchvision
    from mmsr.models import networks
    from mmsr.models.archs.corres_generation_arch import CorrespondenceGenerationArch
    monkeypatch.setenv('C2M_VGG_PRETRAINED', '1')                      # undo the test-suite opt-out
    monkeypatch.setattr(torch.hub, 'get_dir', lambda: str(tmp_path / 'hub'))
    def no_network(*a, **k):
        raise OSError('no network in the test')
    monkeypatch.setattr(torchvision.models, 'vgg19', no_network)
    with pytest.raises(RuntimeError, match='ImageNet weights for vgg19 are not available'):
        CorrespondenceGenerationArch(3, 1, ['relu1_1', 'relu2_1', 'relu3_1'], 'vgg19')
    # a torchvision-format checkpoint (features.N.*) in the hub cache is picked up by the reference YAML's kwargs
    tv = {}
    for n, (ci, co) in zip((0, 2, 5, 7, 10), ((3, 64), (64, 64), (64, 128), (128, 128), (128, 256))):
        tv[f'features.{n}.weight'] = seeding.randn(n + 1, (co, ci, 3, 3))
        tv[f'features.{n}.bias'] = seeding.randn(n + 50, (co,))
    ck = tmp_path / 'hub' / 'checkpoints'
    ck.mkdir(parents=True)
    torch.save(tv, ck / 'vgg19-dcbb9e9d.pth')
    opt = {'network_map': {'type': 'CorrespondenceGenerationArch', 'patch_size': 3, 'stride': 1,
                           'vgg_layer_list': ['relu1_1', 'relu2_1', 'relu3_1'], 'vgg_type': 'vgg19'}}
    net = networks.define_net_map(opt)
    assert torch.equal(net.vgg.vgg_net.conv1_1.weight, tv['features.0.weight'])
    assert torch.equal(net.vgg.vgg_net.conv3_1.bias, tv['features.10.bias'])
    # explicit path / explicit opt-out
    other = tmp_path / 'my_vgg19.pth'
    tv2 = {k: v + 1 for k, v in tv.items()}
    torch.save(tv2, other)
    net2 = CorrespondenceGenerationArch(vgg_pretrained_path=str(other))
    assert torch.equal(net2.vgg.vgg_net.conv2_1.weight, tv2['features.5.weight'])
    net3 = CorrespondenceGenerationArch(vgg_pretrained=False)
    assert not torch.equal(net3.vgg.vgg_net.conv1_1.weight, tv['features.0.weight'])
    with pytest.raises(FileNotFoundError):
        CorrespondenceGenerationArch(vgg_pretrained_path=str(tmp_path / 'missing.pth'))


def test_sharded_eval_sampler_and_shape_buckets():
    """N1: the pair list is partitioned rank::world at the index level (no rank decodes another rank's pairs, nothing
    padded or repeated — unlike the training-side DistIterSampler, data_sampler.py:8-69), and same-shape pairs are
    batched without dropping the ragged tail."""
    from mmsr.data import create_dataloader, create_dataset
    from mmsr.data.data_sampler import ShapeBucketBatchSampler, ShardedEvalSampler
    ds = list(range(126))
    parts = [list(ShardedEvalSampler(ds, 8, r)) for r in range(8)]
    assert sorted(sum(parts, [])) == ds and max(map(len, parts)) - min(map(len, parts)) == 1
    assert parts[3] == list(range(3, 126, 8))
    shapes = {i: ((320, 480) if i % 3 else (336, 496)) for i in parts[3]}
    bs = ShapeBucketBatchSampler(parts[3], shapes.__getitem__, 4)
    got = list(bs)
    assert sorted(sum(got, [])) == parts[3] and all(len({shapes[i] for i in b}) == 1 and len(b) <= 4 for b in got)
    assert len(got) == len(bs)
    # through the factory: synthetic dataset, 2 "ranks", batch 3
    opt = {'name': 'synth', 'type': 'SyntheticRefDataset', 'num': 7, 'gt_size': 32, 'ref_size': 24, 'num_workers': 0,
           'batch_size': 3, 'scale': 4}
    dset = create_dataset(opt)
    seen = []
    for r in range(2):
        loader = create_dataloader(dset, opt, sampler=ShardedEvalSampler(dset, 2, r))
        for batch in loader:
            assert batch['img_in_lq'].shape[1:] == (3, 8, 8) and batch['img_ref'].shape[1:] == (3, 32, 32)
            assert len(batch['lq_path']) == batch['img_in'].shape[0] <= 3
            seen += batch['lq_path']
    assert sorted(seen) == [f'synthetic_{i:04d}.png' for i in range(7)]


def test_pair_batcher_equals_batch_loader():
    """N1: per-sample worker tasks + consumer-side stacking (`PairBatcher`) deliver exactly the batches of the
    per-batch `DataLoader(batch_sampler=...)`, in the same order, with worker processes too."""
    from mmsr.data import PairBatcher, create_dataloader, create_dataset
    opt = {'name': 'synth', 'type': 'SyntheticRefDataset', 'num': 9, 'gt_size': 32, 'ref_size': 24, 'num_workers': 0,
           'batch_size': 4, 'scale': 4}
    dset = create_dataset(opt)
    ref = list(create_dataloader(dset, dict(opt, per_sample_workers=False)))
    for workers in (0, 2):
        loader = create_dataloader(dset, dict(opt, num_workers=workers))
        assert isinstance(loader, PairBatcher) and len(loader) == len(ref) == 3
        assert loader.dataset is dset and loader.batch_sampler.batches == [[0, 1, 2, 3], [4, 5, 6, 7], [8]]
        n = 0
        for got, want in zip(loader, ref):
            for k, v in want.items():
                if torch.is_tensor(v):
                    assert got[k].shape == v.shape and torch.equal(got[k], v), k     # compare before the slot is reused
                else:
                    assert list(got[k]) == list(v), k
            assert ('_slot' in got) == (workers > 0)
            n += 1
        assert n == 3
        if workers:
            # an abandoned pass leaves nothing behind: the next pass starts clean and delivers the same batches
            it = iter(loader)
            next(it)
            it.close()
            again = [b['lq_path'] for b in loader]
            assert again == [list(b['lq_path']) for b in ref]
            loader.close()
            with pytest.raises(RuntimeError, match='closed'):
                next(iter(loader))


def test_pair_batcher_reports_worker_errors_and_mixed_shapes():
    import torch.utils.data as tud
    from mmsr.data import PairBatcher

    class Broken(tud.Dataset):
        opt = {'name': 'broken'}

        def __len__(self):
            return 4

        def __getitem__(self, i):
            if i == 2:
                raise ValueError('cannot decode pair 2')
            return {'img_in': torch.zeros(3, 8 + 4 * (i == 1), 8), 'lq_path': f'{i}.png'}

    loader = PairBatcher(Broken(), [[0], [2]], num_workers=1)
    with pytest.raises(RuntimeError, match='cannot decode pair 2'):
        list(loader)
    loader.close()
    loader = PairBatcher(Broken(), [[0, 1]], num_workers=2)
    with pytest.raises(RuntimeError, match='differ in shape'):
        list(loader)
    loader.close()


def test_metrics_torch_matches_host_metrics():
    """The device-side scores (`metrics_torch.score_image`) follow the reference's metric definitions step by step:
    equal to the numpy / cv2 versions to ~1e-12 incl. crop, un-padding and the non-finite flag."""
    from mmsr.utils import metrics, metrics_torch
    from mmsr.utils.util import tensor2img
    g = torch.Generator().manual_seed(7)
    gt = torch.rand(3, 72, 88, generator=g)
    sr = gt + 0.04 * torch.randn(3, 72, 88, generator=g)
    for crop, valid in ((4, None), (0, None), (4, (66, 81))):
        got = metrics_torch.score_image(sr, gt, crop, valid).tolist()
        a, b = tensor2img([sr, gt])
        if valid:
            a, b = a[:valid[0], :valid[1]], b[:valid[0], :valid[1]]
        ya, yb = metrics.bgr2ycbcr(a / 255., only_y=True), metrics.bgr2ycbcr(b / 255., only_y=True)
        want = (metrics.psnr(a, b, crop_border=crop), metrics.psnr(ya * 255, yb * 255, crop_border=crop),
                metrics.ssim(ya * 255, yb * 255, crop_border=crop))
        assert all(abs(x - y) <= 1e-11 * max(1.0, abs(y)) for x, y in zip(got, want)), (got, want)
        assert got[3] == 1.0
    assert metrics_torch.score_image(gt, gt, 4)[0].item() == float('inf')
    bad = sr.clone()
    bad[1, 5, 5] = float('nan')
    assert metrics_torch.score_image(bad, gt, 4)[3].item() == 0.0


def test_two_product_search_rounding_bound():
    """DESIGN.md K2: the tcgen05 search scores (q_hi + q_lo) . r_hi.  The part of its error that does not come from the
    fp32 accumulation — fp16 rounding of the Ref operand + the query's 22-bit split — stays below
    [2^-11 + 2^-22] ||P_q|| ||P_r||, also for adversarial operands (values just above a rounding midpoint, all products
    of one sign).  Emulated in float64, so the accumulation term is absent by construction."""
    import numpy as np
    rng = np.random.default_rng(3)
    K = 2304

    def split(x, s):
        hi = (x * s).astype(np.float16).astype(np.float64)
        lo = ((x * s) - hi).astype(np.float16).astype(np.float64)
        return hi / s, lo / s

    cases = [(rng.standard_normal(K), rng.standard_normal(K)) for _ in range(40)]
    # adversarial: every Ref element sits just above the midpoint between two fp16 values (relative error -> 2^-11), same sign
    base = 1.0 + 2.0 ** -11 * (1 + 2 * rng.integers(0, 512, K)) + 1e-7
    cases.append((np.abs(rng.standard_normal(K)), base * 2.0 ** rng.integers(-6, 3, K)))
    cases.append((np.ones(K), base))
    worst = 0.0
    for q, r in cases:
        q, r = q.astype(np.float32).astype(np.float64), r.astype(np.float32).astype(np.float64)
        # operands are scaled by a power of two so that amax lands in the fp16 range, as `sexp_kernel` does
        sq = 2.0 ** np.floor(np.log2(2.0 ** 14 / np.abs(q).max()))
        sr = 2.0 ** np.floor(np.log2(2.0 ** 14 / np.abs(r).max()))
        qh, ql = split(q, sq)
        rh, _ = split(r, sr)
        exact = float(np.dot(q, r))
        approx = float(np.dot(qh + ql, rh))
        bound = (2.0 ** -11 + 2.0 ** -22) * np.linalg.norm(q) * np.linalg.norm(r)
        assert abs(approx - exact) <= bound, (abs(approx - exact), bound)
        worst = max(worst, abs(approx - exact) / bound)
    assert 0.0 < worst <= 1.0
    # the window the library uses for K = 2304 (c_abi.cu): 2E for this part, 4E for the accumulation part
    window_coef = 1.01 * 2.0 ** -10 + 2.0 ** -20 * (K / 16 + 3)
    assert window_coef >= 2 * (2.0 ** -11 + 2.0 ** -22 * (K / 16 + 3))
