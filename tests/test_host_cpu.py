"""CPU-side checks of the product: the C-ABI library loads and exports every symbol include/jvae_b200.h declares,
the host mirror builds the same modules / state_dict as the reference (golden fixtures), and compute calls without a
GPU fail loudly (no CPU fallback)."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, golden_names


def test_library_exports_every_declared_symbol(pkg):
    hdr = open(os.path.join(ROOT, 'include', 'jvae_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = sorted(set(re.findall(r'\b(jvae_[a-z0-9_]+)\s*\(', hdr)))
    assert len(declared) >= 15
    lib = ctypes.CDLL(pkg._native.LIB_PATH)
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.jvae_abi_version() == 17


def test_elbo_cfg_struct_matches_header(pkg):
    hdr = open(os.path.join(ROOT, 'include', 'jvae_b200.h')).read()
    body = hdr[hdr.index('typedef struct jvae_elbo_cfg'):hdr.index('} jvae_elbo_cfg;')]
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    fields = []
    for line in body.splitlines()[1:]:
        m = re.match(r'\s*(int32_t|float)\s+([^;]+);', line)
        if m:
            fields += [(n.strip(), m.group(1)) for n in m.group(2).split(',')]
    py = [(n, 'int32_t' if t is ctypes.c_int32 else 'float') for n, t in pkg._native.ElboCfg._fields_]
    assert fields == py


def test_no_cpu_fallback(pkg):
    net = pkg.ClassificationVariationalNetwork((1, 8, 8), 5, type='cvae', encoder=[16], decoder=[16], classifier=[],
                                               latent_dim=8, latent_sampling=2, prior={'var_dim': 'scalar'})
    with pytest.raises(pkg._native.NativeError):
        net.evaluate(torch.rand(4, 1, 8, 8))
    with pytest.raises(pkg._native.NativeError):
        pkg.engine.linear(torch.rand(4, 8), torch.rand(3, 8), None)


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'joint-vae_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'oracle' not in src.replace('the oracle', ''), os.path.join(dirpath, f)


def _ctor_kwargs(cfg):
    kw = json.loads(json.dumps(cfg))
    kw['input_shape'] = tuple(kw['input_shape'])
    return kw


@pytest.mark.parametrize('name', golden_names())
def test_state_dict_matches_reference(pkg, name):
    """same parameter names and shapes as the reference's model (checkpoint contract, SURVEY.md §8b)"""
    d = np.load(os.path.join(GOLDEN, name + '.npz'))
    cfg = json.loads(str(d['cfg']))
    net = pkg.ClassificationVariationalNetwork(**_ctor_kwargs(cfg))
    ref = {k[3:]: d[k].shape for k in d.files if k.startswith('sd.')}
    ours = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert ours == ref
    net.load_state_dict({k: torch.from_numpy(np.asarray(d['sd.' + k])) for k in ours})


@pytest.mark.parametrize('name', golden_names())
def test_layer_stacks_match_reference(pkg, name):
    import importlib.util
    spec = importlib.util.spec_from_file_location('make_golden', os.path.join(GOLDEN, 'make_golden.py'))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    describe = mg.describe
    d = np.load(os.path.join(GOLDEN, name + '.npz'))
    cfg, arch = json.loads(str(d['cfg'])), json.loads(str(d['arch']))
    net = pkg.ClassificationVariationalNetwork(**_ctor_kwargs(cfg))
    assert describe(net.features) == arch['features']
    assert describe(net.encoder.dense_projs) == arch['dense_projs']
    if cfg['type'] != 'vib':
        assert describe(net.decoder) == arch['decoder']
        assert describe(net.imager) == arch['imager']
        assert list(net.imager.input_shape) == arch['imager_in']
    assert net.classifier_type == arch['classifier_type']
    assert bool(net.encoder.sampling.is_sampled) == arch['sampling']


def test_named_presets(pkg):
    conv = pkg.module.vae_layers.conv
    f = conv.build_de_conv_layers((3, 32, 32), 'vgg19', batch_norm=True)
    assert f.output_shape == (512, 1, 1) and f.name == 'vgg19'
    f = conv.build_de_conv_layers((3, 32, 32), 'conv32')
    assert f.output_shape == (200, 2, 2)
    assert conv.find_input_shape('deconv32', (32, 32)) == (1, 1)
    assert conv.find_input_shape('ivgg', (64, 64)) == (4, 4)
    u = conv.build_de_conv_layers((128, 1, 1), 'deconv32', where='output', batch_norm=True)
    assert u.output_shape == (3, 32, 32)
    assert isinstance(u[-1], torch.nn.Identity) and isinstance(u[-2], torch.nn.BatchNorm2d)


def test_prior_api_matches_oracle(pkg):
    """tensor-level prior API (used by callers outside evaluate) against the numpy oracle, on CPU tensors"""
    from oracle import elbo_numpy as on
    pr = pkg.module.priors
    torch.manual_seed(0)
    for var_dim in ('scalar', 'diag', 'full'):
        p = pr.build_prior(8, var_dim=var_dim, num_priors=5, init_mean=1.0, learned_means=True, seed=3)
        with torch.no_grad():
            p._var_parameter.mul_(1 + 0.1 * torch.rand_like(p._var_parameter))
        o = on.Prior(p.mean.detach().numpy(), p._var_parameter.detach().numpy(), var_dim=var_dim)
        mu, lv = torch.randn(6, 8), 0.3 * torch.randn(6, 8)
        y = torch.arange(5)[:, None].repeat(1, 6)
        a = p.kl(mu, lv, y=y, var_weighting=0.7)
        b = o.kl(mu.numpy(), lv.numpy(), y=y.numpy(), var_weighting=0.7)
        for k in ('kl', 'distance', 'var_kl'):
            np.testing.assert_allclose(a[k].detach().numpy(), b[k], rtol=2e-4, atol=1e-4)
        z = torch.randn(3, 5, 6, 8)
        yy = y[None].repeat(3, 1, 1)
        np.testing.assert_allclose(p.log_density(z, yy).detach().numpy(), o.log_density(z.numpy(), yy.numpy()),
                                   rtol=2e-4, atol=1e-4)


def test_losses_api_matches_oracle(pkg):
    from oracle import elbo_numpy as on
    L = pkg.module.losses
    torch.manual_seed(1)
    xo, xt = torch.rand(3, 4, 1, 5, 5), torch.rand(4, 1, 5, 5)
    np.testing.assert_allclose(L.mse_loss(xo, xt, ndim=3, batch_mean=False).numpy(),
                               on.mse_loss(xo.numpy(), xt.numpy(), ndim=3), rtol=1e-5)
    lg = torch.randn(4, 6, 7)
    y = torch.randint(0, 7, (6,))
    np.testing.assert_allclose(L.x_loss(y, lg, batch_mean=False).numpy(), on.x_loss(y.numpy(), lg.numpy()), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(L.x_loss(None, lg, batch_mean=False).numpy(), on.x_loss(None, lg.numpy()), rtol=1e-5, atol=1e-6)
