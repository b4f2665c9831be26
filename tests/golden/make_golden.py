#!/usr/bin/env python
"""Mint the golden fixtures in this directory from the UNMODIFIED reference code.

Needs a checkout of the reference; the tests only read what this script writes:

    python tests/golden/make_golden.py --reference PATH/TO/C2-Matching [corr offsets dcn full dataset specs]

(no fixture names: all of them).  The reference (yumingj/C2-Matching @ 6d60149) ships no tests or
golden vectors (SURVEY.md §4, §8c), so parity is pinned on outputs of the reference's own Python run here
on CPU, imported with three shims that do not touch its arithmetic:
  1. a stub `mmcv` (only `scandir` + the `runner` helpers the imports need),
  2. a stub top-level `_ext` whose `dcn_v2_forward` is torchvision's CPU
     `deform_conv2d(..., mask=...)` — the reference's own `_ext` is CUDA-only and no longer
     compiles (THC removed from torch); oracle/dcn_v2_oracle.c restates its .cu literally
     and tests/test_oracle.py checks the two agree,
  3. `pretrained=False` torchvision VGG constructors (no network).
Inputs and weights come from tests/golden/seeding.py (PCG64), so the tests rebuild them
bit-identically and only OUTPUTS are stored here.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import seeding  # noqa: E402


def install_reference_shims(ref_root):
    import torchvision
    import torchvision.models.vgg as tvgg

    # --- 1. mmcv stub -----------------------------------------------------------------
    mmcv = types.ModuleType('mmcv')

    def scandir(path, suffix=None, recursive=False):
        for f in sorted(os.listdir(path)):
            if suffix is None or f.endswith(suffix):
                yield f

    mmcv.scandir = scandir
    mmcv.mkdir_or_exist = lambda p, mode=0o777: os.makedirs(p, mode=mode, exist_ok=True)
    # image helpers with mmcv 0.4.x semantics (only needed by the dataset fixture)
    import cv2
    mmcv.imfrombytes = lambda content, flag='color': cv2.imdecode(np.frombuffer(content, np.uint8), cv2.IMREAD_COLOR)
    mmcv.bgr2rgb = lambda img: cv2.cvtColor(img, cv2.COLOR_BGR2RGB)

    def impad(img, shape, pad_val=0):
        out = np.full(tuple(shape) + img.shape[2:], pad_val, dtype=img.dtype)
        out[:img.shape[0], :img.shape[1], ...] = img
        return out

    mmcv.impad = impad
    runner = types.ModuleType('mmcv.runner')
    runner.master_only = lambda f: f
    runner.get_dist_info = lambda: (0, 1)
    runner.get_time_str = lambda: 'now'
    runner.init_dist = lambda *a, **k: None
    mmcv.runner = runner
    sys.modules['mmcv'] = mmcv
    sys.modules['mmcv.runner'] = runner

    # --- 2. `_ext` stub ----------------------------------------------------------------
    ext = types.ModuleType('_ext')

    def dcn_v2_forward(input, weight, bias, offset, mask, kh, kw, sh, sw, ph, pw, dh, dw, dg):
        return torchvision.ops.deform_conv2d(
            input, offset, weight, bias, stride=(sh, sw), padding=(ph, pw),
            dilation=(dh, dw), mask=mask)

    ext.dcn_v2_forward = dcn_v2_forward
    sys.modules['_ext'] = ext

    # --- 3. VGG without downloads ------------------------------------------------------
    for name in ('vgg16', 'vgg19'):
        orig = getattr(tvgg, name)

        def make(orig):
            def ctor(pretrained=False, **kw):
                return orig(weights=None)
            return ctor

        setattr(tvgg, name, make(orig))

    sys.path.insert(0, ref_root)


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f'wrote {name}: {os.path.getsize(path) / 1024:.1f} KiB')


# ------------------------------------------------------------------------------------------
CORR_CASES = [
    # name, C, h, w, hr, wr, seed, kind
    ('tiny_c8', 8, 7, 9, 8, 6, 101, 'gauss'),
    ('odd_c32', 32, 13, 11, 17, 19, 102, 'gauss'),
    ('eq_c64', 64, 24, 24, 24, 24, 103, 'gauss'),
    ('planted_c64', 64, 20, 22, 40, 44, 104, 'planted'),
    ('micro_c256', 256, 40, 40, 40, 40, 105, 'gauss'),      # BASELINE config 1 map size
    ('cfg3_c256', 256, 40, 40, 125, 125, 106, 'gauss'),     # BASELINE config 3
    ('min3x3', 16, 3, 3, 3, 3, 107, 'gauss'),               # single patch each side
    ('dup_ref', 16, 6, 6, 10, 10, 108, 'dup'),              # exact ties -> lowest index wins
]


def corr_inputs(case):
    name, c, h, w, hr, wr, seed, kind = case
    if kind == 'gauss':
        return seeding.unit_features(seed, c, h, w), seeding.unit_features(seed + 50, c, hr, wr)
    if kind == 'planted':
        return seeding.planted_features(seed, c, h, w, hr, wr, dy=7, dx=11)
    if kind == 'dup':
        # Ref = a 5x5 block tiled 2x2: every Ref patch fully inside a tile appears 4 times.
        fin = seeding.unit_features(seed, c, h, w)
        blk = seeding.unit_features(seed + 50, c, 5, 5)
        return fin, blk.repeat(1, 2, 2)
    raise ValueError(kind)


def gen_corr():
    from mmsr.models.archs.ref_map_util import feature_match_index
    out = {}
    for case in CORR_CASES:
        name = case[0]
        fin, fref = corr_inputs(case)
        for norm_input in (True, False):
            idx, val = feature_match_index(fin, fref, 3, 1, 1, is_norm=True, norm_input=norm_input)
            tag = f'{name}/ni{int(norm_input)}'
            out[tag + '/idx'] = idx.numpy().astype(np.int32)
            out[tag + '/val'] = val.numpy()
        # fp64 run of the same reference code: tie/margin analysis
        idx64, _ = feature_match_index(fin.double(), fref.double(), 3, 1, 1, True, True)
        out[name + '/idx64'] = idx64.numpy().astype(np.int32)
        out[name + '/sha_in'] = np.array(seeding.sha(fin))
        out[name + '/sha_ref'] = np.array(seeding.sha(fref))
        agree = bool((idx64 == idx).all())
        print(f'  corr {name}: fp32==fp64 idx: {agree}')
    # is_norm=False flavour on one case (API coverage)
    fin, fref = corr_inputs(CORR_CASES[1])
    idx, val = feature_match_index(fin, fref, 3, 1, 1, is_norm=False, norm_input=False)
    out['odd_c32/raw/idx'] = idx.numpy().astype(np.int32)
    out['odd_c32/raw/val'] = val.numpy()
    save('corr.npz', **out)


def gen_offsets():
    """pre_offset pyramids from the reference CorrespondenceGenerationArch.forward
    (corres_generation_arch.py:48-117) on small seeded feature maps, B=2."""
    from mmsr.models.archs.corres_generation_arch import CorrespondenceGenerationArch
    net = CorrespondenceGenerationArch(3, 1, ['relu1_1', 'relu2_1', 'relu3_1'], 'vgg19').eval()
    seeding.fill_state_dict_(net, 7)
    out = {}
    for tag, (c, h, w) in {'a': (32, 12, 12), 'b': (16, 9, 14)}.items():
        f1 = seeding.randn(300 + ord(tag), (2, c, h, w))
        f2 = seeding.randn(400 + ord(tag), (2, c, h, w))
        img_ref = seeding.rand_image(500 + ord(tag), (2, 3, 4 * h, 4 * w))
        with torch.no_grad():
            pre, feats = net({'dense_features1': f1, 'dense_features2': f2}, img_ref)
        for k, v in pre.items():
            assert torch.equal(v, v.round())
            out[f'{tag}/{k}'] = v.numpy().astype(np.int16)
        out[f'{tag}/relu3_1_sum'] = np.array(float(feats['relu3_1'].double().sum()))
    save('offsets.npz', **out)


DCN_CASES = [
    # name, B, C, Cout, H, W, dg, seed, offset_scale
    ('small', 2, 16, 16, 12, 10, 4, 201, 1.0),
    ('wide', 1, 64, 64, 20, 24, 8, 202, 3.0),
    ('ragged', 1, 24, 40, 7, 13, 8, 203, 6.0),     # C/dg = 3, Cout != C, offsets leave the image
]


def dcn_inputs(case):
    name, b, c, cout, h, w, dg, seed, osc = case
    x = seeding.randn(seed, (b, c, h, w))
    feat = seeding.randn(seed + 1, (b, c, h, w))
    rng = np.random.default_rng(seed + 2)
    pre = torch.from_numpy(rng.integers(-int(4 * osc), int(4 * osc) + 1, (b, 9, h, w, 2)).astype(np.float32))
    return x, feat, pre


def gen_dcn():
    from mmsr.models.archs.DCNv2.dcn_v2 import DCN_sep_pre_multi_offset
    out = {}
    for case in DCN_CASES:
        name, b, c, cout, h, w, dg, seed, osc = case
        m = DCN_sep_pre_multi_offset(c, cout, 3, stride=1, padding=1, dilation=1,
                                     deformable_groups=dg, extra_offset_mask=True).eval()
        seeding.fill_state_dict_(m, seed + 3)
        with torch.no_grad():
            m.conv_offset_mask.weight.mul_(osc)
        x, feat, pre = dcn_inputs(case)
        with torch.no_grad():
            y = m([x, feat], pre)
        out[name + '/out'] = y.numpy()
    save('dcn.npz', **out)


def gen_full():
    """BASELINE config 1: LR 40x40, Ref 64x64 zero-padded to 160x160, B=1, full forward
    (extractor -> net_map -> net_g) through the reference classes."""
    from mmsr.models.archs.contras_extractor_arch import ContrasExtractorSep
    from mmsr.models.archs.corres_generation_arch import CorrespondenceGenerationArch
    from mmsr.models.archs.ref_restoration_arch import RestorationNet
    import mmsr.models.archs.corres_generation_arch as cga

    ext = ContrasExtractorSep().eval()
    net_map = CorrespondenceGenerationArch(3, 1, ['relu1_1', 'relu2_1', 'relu3_1'], 'vgg19').eval()
    net_g = RestorationNet(ngf=64, n_blocks=16, groups=8).eval()
    seeding.fill_state_dict_(ext, 11)
    ext.load_state_dict(seeding.share_extractor_weights(ext.state_dict()))
    seeding.fill_state_dict_(net_map, 12)
    seeding.fill_state_dict_(net_g, 13)

    from oracle import c_oracle
    out = {}
    for tag in ('cfg1', 'b2'):
        hr, img_lq, img_up, img_ref = seeding.full_case_inputs(tag)
        grabbed = []
        orig = cga.feature_match_index

        def spy(*a, **k):
            r = orig(*a, **k)
            grabbed.append(r[0].clone())
            return r

        cga.feature_match_index = spy
        try:
            with torch.no_grad():
                feats = ext(img_up, img_ref)
                pre, ref_feat = net_map(feats, img_ref)
                sr = net_g(img_lq, pre, ref_feat)
        finally:
            cga.feature_match_index = orig
        out[tag + '/sr'] = sr.numpy()
        out[tag + '/max_idx'] = torch.stack(grabbed).numpy().astype(np.int32)
        # fp64 top-1/top-2 margins of every query (literal C oracle on the reference's features)
        gaps = []
        for bi in range(img_lq.shape[0]):
            c, h, w = feats['dense_features1'][bi].shape
            a = F.normalize(feats['dense_features1'][bi].reshape(c, -1), dim=0).view(c, h, w)
            r = F.normalize(feats['dense_features2'][bi].reshape(c, -1), dim=0).view(c, h, w)
            oi, _, gp = c_oracle.corr_argmax(a, r, is_norm=True, norm_input=True, want_gap=True)
            assert torch.equal(oi, grabbed[bi])
            gaps.append(gp)
        out[tag + '/gap64'] = torch.stack(gaps).numpy()
        print(f'  full {tag}: min gap {float(torch.stack(gaps).min()):.3e}, #gap<1e-4: {int((torch.stack(gaps) < 1e-4).sum())}')
        out[tag + '/feat1_sum'] = np.array(float(feats['dense_features1'].double().sum()))
        print(f'  full {tag}: sr mean {sr.mean():.5f} std {sr.std():.5f}')
    save('full.npz', **out)


def dataset_pngs(root):
    """Two deterministic (input, ref) PNG pairs with sizes that exercise mod-crop and both padding directions."""
    import cv2
    os.makedirs(root, exist_ok=True)
    specs = [('a', (70, 94), (53, 41)), ('b', (48, 40), (66, 90))]      # (H, W) input / ref
    lines = []
    for tag, (ih, iw), (rh, rw) in specs:
        for kind, (h, w), seed in (('in', (ih, iw), 1), ('ref', (rh, rw), 2)):
            img = (seeding.structured_image(ord(tag) * 10 + seed, 1, max(h, w))[0, :, :h, :w].permute(1, 2, 0).numpy() * 255).round().astype(np.uint8)
            cv2.imwrite(os.path.join(root, f'{tag}_{kind}.png'), img)
        lines.append(f'{tag}_in.png {tag}_ref.png')
    with open(os.path.join(root, 'pairs.txt'), 'w') as f:
        f.write('\n'.join(lines) + '\n')
    return os.path.join(root, 'pairs.txt')


def gen_dataset():
    """Test-phase samples of the reference RefCUFEDDataset (mmsr/data/ref_cufed_dataset.py:63-167)."""
    import tempfile
    from mmsr.data.ref_cufed_dataset import RefCUFEDDataset
    out = {}
    with tempfile.TemporaryDirectory() as root:
        ann = dataset_pngs(root)
        ds = RefCUFEDDataset({'dataroot_in': root, 'dataroot_ref': root, 'ann_file': ann, 'io_backend': {'type': 'disk'},
                              'scale': 4, 'phase': 'test', 'name': 'g'})
        for i in range(len(ds)):
            s = ds[i]
            for k in ('img_in', 'img_in_lq', 'img_in_up', 'img_ref', 'img_ref_lq', 'img_ref_up'):
                out[f'{i}/{k}'] = s[k].numpy()
            out[f'{i}/padding'] = np.array(bool(s['padding']))
            out[f'{i}/original_size'] = np.array(s['original_size'])
    save('dataset.npz', **out)


def gen_specs():
    """State-dict key -> shape of the three reference nets as the model builds them, for the hand-written
    specs in seeding.py (RestorationNet(64, 16, 8), ContrasExtractorSep(), CorrespondenceGenerationArch(vgg19))."""
    import json
    from mmsr.models.archs.contras_extractor_arch import ContrasExtractorSep
    from mmsr.models.archs.corres_generation_arch import CorrespondenceGenerationArch
    from mmsr.models.archs.ref_restoration_arch import RestorationNet
    out = {}
    for n, net in (('g', RestorationNet(64, 16, 8)), ('e', ContrasExtractorSep()),
                   ('m', CorrespondenceGenerationArch(3, 1, ['relu1_1', 'relu2_1', 'relu3_1'], 'vgg19'))):
        out[n] = {k: list(v.shape) for k, v in net.state_dict().items()}
    # one `"key": [shape]` entry per line, so that a change of the specs reads as a change of the lines it touches
    nets = []
    for n, spec in out.items():
        entries = ',\n'.join(f'  {json.dumps(k)}: {json.dumps(v)}' for k, v in spec.items())
        nets.append(f' {json.dumps(n)}: {{\n{entries}\n }}')
    path = os.path.join(HERE, 'reference_specs.json')
    with open(path, 'w') as f:
        f.write('{\n' + ',\n'.join(nets) + '\n}\n')
    print(f'wrote reference_specs.json: {os.path.getsize(path) / 1024:.1f} KiB')


GENERATORS = {'corr': gen_corr, 'offsets': gen_offsets, 'dcn': gen_dcn, 'full': gen_full, 'dataset': gen_dataset,
              'specs': gen_specs}


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument('--reference', required=True, help='checkout of yumingj/C2-Matching @ 6d60149')
    ap.add_argument('fixtures', nargs='*', help=f'any of {" ".join(GENERATORS)} (default: all)')
    args = ap.parse_args()
    unknown = set(args.fixtures) - set(GENERATORS)
    if unknown:
        ap.error(f'unknown fixtures: {sorted(unknown)}')
    torch.manual_seed(0)
    torch.set_num_threads(8)
    install_reference_shims(args.reference)
    names = args.fixtures or list(GENERATORS)
    for name in names:
        GENERATORS[name]()
    # VERSIONS.txt stamps every stored fixture, so it is only rewritten when all of them were regenerated
    if set(names) == set(GENERATORS):
        meta = f'torch {torch.__version__}; numpy {np.__version__}; reference 6d60149\n'
        with open(os.path.join(HERE, 'VERSIONS.txt'), 'w') as f:
            f.write(meta)
    else:
        print('VERSIONS.txt left as is: it records the versions of the last full regeneration')


if __name__ == '__main__':
    main()
