"""Deterministic synthetic weights / inputs shared by the golden generator and the tests.

Everything is drawn from numpy's PCG64 (`np.random.default_rng`), whose stream is
stable across numpy versions and machines, so the same tensors are rebuilt on the GPU
box without shipping them.  The reference nets and the B200 nets share state-dict keys
(SURVEY.md §5 "checkpoint"), so filling by *sorted key* gives both the same weights.
"""
import hashlib

import numpy as np
import torch


def _gain_for(key: str) -> float:
    # ResBlock bodies: small residual branch, like the reference's default_init_weights(…, 0.1)
    # (mmsr/models/archs/arch_util.py:40-61); everything else unit-gain He-style.
    if '.body' in key or key.startswith('body') or 'content_extractor.body' in key:
        return 0.1 * np.sqrt(2.0)
    if 'vgg' in key or 'feature_extraction' in key:
        return np.sqrt(2.0)
    return 1.0


def fill_state_dict_(module: torch.nn.Module, seed: int) -> None:
    """In-place: overwrite every floating parameter of `module` from PCG64(seed)."""
    rng = np.random.default_rng(seed)
    sd = module.state_dict()
    for key in sorted(sd.keys()):
        t = sd[key]
        if not t.is_floating_point():
            continue
        if key.endswith('mean') or key.endswith('std'):
            continue  # ImageNet normalisation buffers stay as constructed
        shape = tuple(t.shape)
        if t.dim() >= 2:
            fan_in = int(np.prod(shape[1:]))
            v = rng.standard_normal(shape) * (_gain_for(key) / np.sqrt(fan_in))
        else:
            v = rng.standard_normal(shape) * 0.1
        t.copy_(torch.from_numpy(v.astype(np.float32)))


def structured_image(seed: int, batch: int, n: int) -> torch.Tensor:
    """Multi-scale block texture in [0,1], [batch,3,n,n]: unlike iid noise it gives feature maps with
    position-dependent content, so the correspondence search is well conditioned (top-1/top-2
    margins far above fp32 noise)."""
    out = []
    for b in range(batch):
        rng = np.random.default_rng(seed * 1000 + b)
        img = np.zeros((3, n, n))
        for s in (2, 4, 8, 16):
            m = n // s + 1
            img += np.kron(rng.random((3, m, m)), np.ones((1, s, s)))[:, :n, :n] * (s / 30.0)
        out.append(img / img.max())
    return torch.from_numpy(np.stack(out).astype(np.float32))


def share_extractor_weights(sd: dict) -> dict:
    """Give both ContrasExtractor trunks the same weights.  The trained reference checkpoint has two
    trunks trained to be mutually compatible; two independent RANDOM trunks would make every
    LR<->Ref correlation pure noise (argmax decided at the 1e-6 level)."""
    for k in list(sd):
        if k.startswith('feature_extraction_image2.model'):
            sd[k] = sd[k.replace('image2', 'image1')].clone()
    return sd


def full_case_inputs(tag: str):
    """Inputs of the full-forward golden cases (make_golden.gen_full and the tests)."""
    import torch.nn.functional as F
    b, lr, refsz, seed = {'cfg1': (1, 40, 64, 21), 'b2': (2, 24, 40, 22)}[tag]
    hr = structured_image(seed, b, 4 * lr)
    img_lq = F.interpolate(hr, scale_factor=0.25, mode='bicubic', align_corners=False).clamp(0, 1)
    img_up = F.interpolate(img_lq, scale_factor=4, mode='bicubic', align_corners=False).clamp(0, 1)
    if tag == 'cfg1':      # Ref shares content with the input: a shifted crop of the HR image
        ref = hr[:, :, 16:16 + refsz, 24:24 + refsz].clone()
    else:                  # unrelated Ref
        ref = structured_image(seed + 1, b, refsz)
    img_ref = F.pad(ref, (0, 4 * lr - refsz, 0, 4 * lr - refsz))
    return hr, img_lq, img_up, img_ref


def rand_image(seed: int, shape) -> torch.Tensor:
    """U[0,1) image batch, float32 NCHW."""
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.random(shape, dtype=np.float64).astype(np.float32))


def randn(seed: int, shape, scale: float = 1.0) -> torch.Tensor:
    rng = np.random.default_rng(seed)
    return torch.from_numpy((rng.standard_normal(shape) * scale).astype(np.float32))


def unit_features(seed: int, c: int, h: int, w: int) -> torch.Tensor:
    """SURVEY.md §8(d) config 3: per-pixel channel-unit-norm Gaussian feature map [c,h,w]."""
    x = randn(seed, (c, h, w)).double()
    x = x / x.norm(dim=0, keepdim=True).clamp_min(1e-12)
    return x.float()


def planted_features(seed: int, c: int, h: int, w: int, hr: int, wr: int, dy: int, dx: int,
                     noise: float = 0.05):
    """Planted-match pair: the input map is a crop of the Ref map at (dy,dx) plus small noise,
    so argmax must recover a pure translation for interior patches."""
    ref = randn(seed, (c, hr, wr))
    inp = ref[:, dy:dy + h, dx:dx + w] + randn(seed + 1, (c, h, w), noise)
    nrm = lambda t: (t.double() / t.double().norm(dim=0, keepdim=True).clamp_min(1e-12)).float()
    return nrm(inp), nrm(ref)


def sha(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()[:16]


# --------------------------------------------------------------------------------------------
# State-dict specifications (key -> shape) of the three reference nets, written out by hand from
# the reference constructors so that neither the oracle tests nor the GPU box need the reference:
#   RestorationNet(ngf=64, n_blocks=16, groups=8)   mmsr/models/archs/ref_restoration_arch.py:30-145
#   ContrasExtractorSep()                            mmsr/models/archs/contras_extractor_arch.py:8-59
#   CorrespondenceGenerationArch(vgg19, relu3_1)     mmsr/models/archs/corres_generation_arch.py:14-27
# tests/test_host_cpu.py checks them against the reference classes' state dicts (reference_specs.json).
def _conv_spec(d, name, cin, cout, k=3):
    d[name + '.weight'] = (cout, cin, k, k)
    d[name + '.bias'] = (cout,)


def _body_spec(d, name, n, nf):
    for i in range(n):
        _conv_spec(d, f'{name}.{i}.conv1', nf, nf)
        _conv_spec(d, f'{name}.{i}.conv2', nf, nf)


def spec_restoration_net(ngf=64, n_blocks=16, groups=8):
    d = {}
    _conv_spec(d, 'content_extractor.conv_first', 3, ngf)
    _body_spec(d, 'content_extractor.body', n_blocks, ngf)
    p = 'dyn_agg_restore.'
    for size, c in (('small', 256), ('medium', 128), ('large', 64)):
        _conv_spec(d, f'{p}{size}_offset_conv1', ngf + c, c)
        _conv_spec(d, f'{p}{size}_offset_conv2', c, c)
        d[f'{p}{size}_dyn_agg.weight'] = (c, c, 3, 3)
        d[f'{p}{size}_dyn_agg.bias'] = (c,)
        _conv_spec(d, f'{p}{size}_dyn_agg.conv_offset_mask', c, groups * 27)
        _conv_spec(d, f'{p}head_{size}.0', ngf + c, ngf)
        _body_spec(d, f'{p}body_{size}', n_blocks, ngf)
    _conv_spec(d, f'{p}tail_small.0', ngf, ngf * 4)
    _conv_spec(d, f'{p}tail_medium.0', ngf, ngf * 4)
    _conv_spec(d, f'{p}tail_large.0', ngf, ngf // 2)
    _conv_spec(d, f'{p}tail_large.2', ngf // 2, 3)
    return d


_VGG_TO_3_1 = (('conv1_1', 3, 64), ('conv1_2', 64, 64), ('conv2_1', 64, 128), ('conv2_2', 128, 128),
               ('conv3_1', 128, 256))


def spec_extractor():
    d = {}
    for owner in ('feature_extraction_image1', 'feature_extraction_image2'):
        for n, ci, co in _VGG_TO_3_1:
            _conv_spec(d, f'{owner}.model.{n}', ci, co)
        d[owner + '.mean'] = (1, 3, 1, 1)
        d[owner + '.std'] = (1, 3, 1, 1)
    return d


def spec_net_map():
    d = {}
    for n, ci, co in _VGG_TO_3_1:
        _conv_spec(d, f'vgg.vgg_net.{n}', ci, co)
    d['vgg.mean'] = (1, 3, 1, 1)
    d['vgg.std'] = (1, 3, 1, 1)
    return d


_IMAGENET_MEAN = (0.485, 0.456, 0.406)
_IMAGENET_STD = (0.229, 0.224, 0.225)


def seeded_state_dict(spec: dict, seed: int) -> dict:
    """Same stream as fill_state_dict_(module, seed) for a module whose state dict == spec."""
    rng = np.random.default_rng(seed)
    sd = {}
    for key in sorted(spec.keys()):
        shape = tuple(spec[key])
        if key.endswith('mean'):
            sd[key] = torch.tensor(_IMAGENET_MEAN).view(1, 3, 1, 1)
            continue
        if key.endswith('std'):
            sd[key] = torch.tensor(_IMAGENET_STD).view(1, 3, 1, 1)
            continue
        if len(shape) >= 2:
            fan_in = int(np.prod(shape[1:]))
            v = rng.standard_normal(shape) * (_gain_for(key) / np.sqrt(fan_in))
        else:
            v = rng.standard_normal(shape) * 0.1
        sd[key] = torch.from_numpy(v.astype(np.float32))
    return sd
