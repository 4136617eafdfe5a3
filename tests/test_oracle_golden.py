"""Pins oracle/nero_oracle.py to the golden vectors produced by the UNMODIFIED reference
(oracle/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest
import torch

import nero_oracle as O
import nero_oracle_mat as OM
from helpers import load_golden, build_params, param_checksums, t, rays_from_golden, FIXTURE_CFGS, FIXTURE_STEPS, VAL_FIXTURES
from helpers import MATERIAL_FIXTURES, build_material_params, material_batch_from_golden, material_rands

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_encoding_kats():
    g = load_golden('kat_encodings')
    x = t(g['x'])
    for L in (4, 6, 8):
        assert torch.equal(O.embed(x, L), t(g[f'pe{L}']))
    assert torch.equal(O.embed(t(g['x4']), 10), t(g['pe10_4']))
    ide = O.ide(t(g['ide_dirs']), t(g['ide_kappa']))
    np.testing.assert_allclose(ide.numpy(), g['ide'], rtol=0, atol=1e-6)
    assert torch.equal(O.ipe(t(g['ipe_mean']), t(g['ipe_var']), 0, 6), t(g['ipe']))
    assert torch.equal(O.linear_to_srgb(t(g['srgb_in'])), t(g['srgb']))
    assert torch.equal(O.sample_pdf(t(g['pdf_bins']), t(g['pdf_w']), 16), t(g['pdf_out']))


def test_known_answers_from_survey():
    # SURVEY.md Appendix D
    pe = O.embed(torch.tensor([[0.1, 0.2, 0.3]]), 6)[0]
    np.testing.assert_allclose(pe[:9].numpy(), [0.1, 0.2, 0.3, 0.0998, 0.1987, 0.2955, 0.9950, 0.9801, 0.9553], atol=1e-4)
    d = torch.nn.functional.normalize(torch.tensor([[1e-6, 1e-6, 1.0]]), dim=-1)
    e = O.ide(d, torch.zeros(1, 1))[0]
    np.testing.assert_allclose(e[[0, 2, 5, 10, 19]].numpy(), [0.4886, 0.6308, 0.8463, 1.1631, 1.6221], atol=2e-4)
    lut = torch.from_numpy(np.fromfile(os.path.join(ROOT, 'assets', 'bsdf_256_256.bin'), dtype=np.float32).reshape(256, 256, 2).copy())
    # LUT corner KATs: uv = [NoV, roughness] -> lut[row=roughness, col=NoV]
    for uv, want in [((0.0, 0.0), (0.00972746, 0.9902487)), ((1.0, 0.0), (1.0, 2.84e-14)),
                     ((0.0, 1.0), (0.941525, 0.04653827)), ((1.0, 1.0), (0.30927664, 3.5468642e-05))]:
        got = O.fg_lookup(lut, torch.tensor([uv]))[0]
        np.testing.assert_allclose(got.numpy(), want, rtol=1e-5, atol=1e-9)
    # texel centre -> exact texel
    got = O.fg_lookup(lut, torch.tensor([[(10 + 0.5) / 256, (20 + 0.5) / 256]]))[0]
    np.testing.assert_allclose(got.numpy(), lut[20, 10].numpy(), rtol=1e-6)


@pytest.mark.parametrize('name', list(FIXTURE_CFGS))
def test_shape_fixture(name):
    g = load_golden(name)
    cfg = FIXTURE_CFGS[name]
    sd = build_params(cfg, int(g['seed']), int(g['pseed']))
    np.testing.assert_allclose(param_checksums(sd), g['param_checksums'], rtol=1e-12)
    rays = rays_from_golden(g)
    c = O.merged_cfg(cfg)
    lut = sd['color_network.FG_LUT'][0]
    with torch.no_grad():
        z = O.sample_ray(sd, c, rays['rays_o'], rays['rays_d'], rays['near'], rays['far'])
        zp = O.sample_ray(sd, c, rays['rays_o'], rays['rays_d'], rays['near'], rays['far'], t(g['rand_inner']), t(g['rand_bg']))
    assert torch.equal(z, t(g['z_vals']))
    assert torch.equal(zp, t(g['z_vals_perturbed']))
    names = [str(n) for n in g['param_names']]
    for step in FIXTURE_STEPS[name]:
        p = {k: v.clone().requires_grad_(k in names) for k, v in sd.items()}
        out = O.render_core(p, c, lut, rays['rays_o'], rays['rays_d'], z, rays['human_poses'], O.get_anneal_val(c, step), step)
        loss = O.training_loss(out, rays['rgb'], c, step)
        loss.backward()
        pre = f's{step}_'
        for k in ('ray_rgb', 'gradient_error', 'std', 'loss_occ'):
            np.testing.assert_allclose(out[k].detach().numpy().reshape(-1), g[pre + k].reshape(-1), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(float(loss), float(g[pre + 'loss']), rtol=1e-6)
        gn = np.array([float(p[n].grad.double().norm()) if p[n].grad is not None else 0.0 for n in names])
        np.testing.assert_allclose(gn, g[pre + 'grad_norms'], rtol=1e-4, atol=1e-9)
        for k in g:
            if k.startswith(pre + 'grad::'):
                np.testing.assert_allclose(p[k.split('::')[1]].grad.numpy(), g[k], rtol=1e-4, atol=1e-7)


def test_materials_field_and_pole_fixtures():
    """Round-2 fixtures of the unmodified reference: color_network.predict_materials on sdf_network features
    (renderer.py:629-647), the extract_fields grid (field.py:1090-1104) and the IDE near the poles."""
    g = load_golden('shape_materials_field')
    cfg = {'n_samples': 32, 'n_importance': 32}
    sd = build_params(cfg, int(g['seed']), int(g['pseed']))
    np.testing.assert_allclose(param_checksums(sd), g['param_checksums'], rtol=1e-12)
    xyz = t(g['xyz'])
    with torch.no_grad():
        y = O.sdf_forward(sd, xyz)
        fin = torch.cat([y[:, 1:], xyz], -1)
        for k in ('metallic', 'roughness', 'albedo'):
            got = O.predictor(sd, f'color_network.{k}_predictor', fin, 'sigmoid')
            np.testing.assert_allclose(got.numpy(), g[k], rtol=1e-5, atol=1e-6, err_msg=k)
        ax = torch.linspace(-1, 1, 24)
        pts = torch.stack(torch.meshgrid(ax, ax, ax, indexing='ij'), -1).reshape(-1, 3)
        val = O.sdf_forward(sd, pts)[:, 0]
        val = torch.where(torch.norm(pts, dim=-1) >= 1.0, torch.ones_like(val), val).reshape(24, 24, 24)
    np.testing.assert_allclose(val.numpy(), g['field24'], rtol=1e-5, atol=2e-6)
    gp = load_golden('kat_ide_poles')
    np.testing.assert_allclose(O.ide(t(gp['dirs']), t(gp['kappa'])).numpy(), gp['ide'], rtol=0, atol=1e-6)


@pytest.mark.parametrize('name', list(VAL_FIXTURES))
def test_validation_fixture(name):
    """is_train=False render (network/renderer.py:465-482) of the oracle vs the unmodified reference."""
    g = load_golden(name)
    cfg = VAL_FIXTURES[name]
    sd = build_params(cfg, int(g['seed']), int(g['pseed']))
    np.testing.assert_allclose(param_checksums(sd), g['param_checksums'], rtol=1e-12)
    rays = O.synthetic_rays(int(g['R']), seed=int(g['seed']))
    c = O.merged_cfg(cfg)
    step = int(g['step'])
    with torch.no_grad():
        out = O.render_core(sd, c, sd['color_network.FG_LUT'][0], rays['rays_o'], rays['rays_d'], t(g['z_vals']), rays['human_poses'],
                            O.get_anneal_val(c, step), step, is_train=False)
    keys = [k[4:] for k in g if k.startswith('val_')]
    assert set(keys) == set(out.keys())
    for k in keys:
        np.testing.assert_allclose(out[k].numpy().reshape(-1), g['val_' + k].reshape(-1), rtol=2e-5, atol=2e-6, err_msg=k)


@pytest.mark.parametrize('name', list(MATERIAL_FIXTURES))
def test_material_fixture(name):
    """Stage II oracle (MCShadingNetwork + train-step glue) vs the unmodified reference, same tracer, same random draws."""
    g = load_golden(name)
    cfg, steps = MATERIAL_FIXTURES[name]
    scfg = cfg['shader_cfg']
    sd = build_material_params(scfg, int(g['seed']), int(g['pseed']))
    np.testing.assert_allclose(param_checksums(sd), g['param_checksums'], rtol=1e-12)
    verts, tris = OM.test_scene(2)
    trace_fn = lambda o, d: OM.renderer_trace(verts, tris, o, d)
    batch = material_batch_from_golden(g)
    again = OM.synthetic_surface_batch(verts, tris, int(g['P']), seed=int(g['seed']))
    assert all(torch.equal(batch[k], again[k]) for k in batch)
    tabs = (OM.direction_samples(scfg['diffuse_sample_num']), OM.direction_samples(scfg['specular_sample_num']))
    names = [str(n) for n in g['param_names']]
    for step in steps:
        p = {k: v.clone().requires_grad_(k in names) for k, v in sd.items()}
        out = OM.material_train_outputs(p, cfg, tabs, trace_fn, batch, step, material_rands(g, step))
        loss = OM.material_training_loss(out)
        loss.backward()
        pre = f's{step}_'
        for k in out:
            np.testing.assert_allclose(out[k].detach().numpy().reshape(-1), g[pre + k].reshape(-1), rtol=2e-5, atol=2e-6, err_msg=k)
        np.testing.assert_allclose(float(loss), float(g[pre + 'loss']), rtol=1e-6)
        gn = np.array([float(p[n].grad.double().norm()) if p[n].grad is not None else 0.0 for n in names])
        np.testing.assert_allclose(gn, g[pre + 'grad_norms'], rtol=2e-4, atol=1e-9)
        for k in g:
            if k.startswith(pre + 'grad::'):
                np.testing.assert_allclose(p[k.split('::')[1]].grad.numpy(), g[k], rtol=2e-4, atol=1e-7)
