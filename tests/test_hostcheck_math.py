"""CPU check of the hand-derived per-sample math (nero_b200/csrc/math_*.cuh compiled for the HOST by nvcc)
against the oracle (values) and the oracle's autograd in float64 (gradients)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

import nero_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'hostcheck', 'hostcheck.cu')
SO = os.path.join(HERE, 'hostcheck', 'libhostcheck.so')


@pytest.fixture(scope='module')
def hc():
    deps = [SRC] + [os.path.join(HERE, '..', 'nero_b200', 'csrc', f) for f in ('math_enc.cuh', 'math_shade.cuh', 'math_mc.cuh', 'common.cuh')]
    if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in deps):
        subprocess.check_call(['/usr/local/cuda/bin/nvcc', '-O2', '-std=c++17', '-Xcompiler', '-fPIC', '-shared', '--fmad=false',
                               '-Wno-deprecated-gpu-targets', '-o', SO, SRC])
    lib = ctypes.CDLL(SO)
    _, mat = O.ide_tables(5)
    lib.hc_set_ide(np.ascontiguousarray(mat, dtype=np.float32).ctypes.data_as(ctypes.c_void_p))
    return lib


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def f32(x):
    return np.ascontiguousarray(x.detach().numpy() if torch.is_tensor(x) else x, dtype=np.float32)


def close(got, want, rtol, atol, name=''):
    want = want.detach().numpy() if torch.is_tensor(want) else want
    err = np.abs(got - want) - (atol + rtol * np.abs(want))
    assert err.max() <= 0, f'{name}: max violation {err.max():.3e} (abs err {np.abs(got - want).max():.3e})'


def test_ide(hc):
    g = torch.Generator().manual_seed(3)
    n = 400
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    kap = torch.rand(n, 1, generator=g)
    kap[:50] = 0
    dout = torch.randn(n, 72, generator=g)
    dd = d.double().requires_grad_(True)
    kk = kap.double().requires_grad_(True)
    want = O.ide(dd, kk)
    (want * dout.double()).sum().backward()
    out, gd, gk = np.zeros((n, 72), np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
    hc.hc_ide(n, P(f32(d)), P(f32(kap[:, 0])), P(f32(dout)), P(out), P(gd), P(gk))
    # the VALUE follows the reference's own fp32 arithmetic (correctly rounded z powers, ascending FMA chain; math_enc.cuh):
    # it agrees with the fp32 oracle (bit-exact to the reference) to the rounding of the (x+iy)^m recurrence and expf, and
    # therefore carries the reference's l=16 cancellation error against exact arithmetic
    w32 = O.ide(d, kap)
    # (residual: torch evaluates (x+iy)^m as exp(m log z) in fp32, 4e-6 absolute away from the exact power; the kernel's
    # recurrence is accurate to 3e-7 -- measured in round 2)
    close(out, w32, 1e-5, 1.2e-5, 'ide value vs the reference arithmetic')
    assert np.abs(out - want.detach().numpy()).max() < 2e-2
    close(gd, dd.grad, 1e-4, 5e-4, 'ide d/ddir')
    close(gk, kk.grad[:, 0], 1e-4, 5e-4, 'ide d/dkappa')


def test_ide_near_the_poles_matches_the_reference(hc):
    """Directions within 1e-4 .. 5e-2 of +-z, roughness 0 / 0.3 / 1: the l = 16 band of the reference is up to 2.4e-3 away
    from exact arithmetic there (fixture from the unmodified reference, oracle/make_golden.py --round2-only)."""
    from helpers import load_golden
    gp = load_golden('kat_ide_poles')
    n = gp['dirs'].shape[0]
    out, gd, gk = np.zeros((n, 72), np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
    dout = np.zeros((n, 72), np.float32)
    hc.hc_ide(n, P(f32(gp['dirs'])), P(f32(gp['kappa'][:, 0])), P(dout), P(out), P(gd), P(gk))
    close(out, gp['ide'], 1e-5, 1.2e-5, 'ide at the poles vs the reference')
    exact = O.ide(torch.from_numpy(gp['dirs']).double(), torch.from_numpy(gp['kappa']).double()).numpy()
    assert np.abs(gp['ide'] - exact).max() > 1e-3, 'the fixture must exercise the cancellation regime'


def test_pe(hc):
    g = torch.Generator().manual_seed(4)
    n, L = 100, 6
    x = torch.rand(n, 3, generator=g) * 2 - 1
    u = torch.randn(n, 39, generator=g)
    dv = torch.randn(n, 3, generator=g)
    xd = x.double().requires_grad_(True)
    pe = O.embed(xd, L)
    (pe * u.double()).sum().backward()
    jt = torch.autograd.functional.jvp(lambda a: O.embed(a, L), x.double(), dv.double())[1]
    o_pe, o_g, o_t = np.zeros((n, 39), np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 39), np.float32)
    hc.hc_pe(n, L, P(f32(x)), P(f32(u)), P(f32(dv)), P(o_pe), P(o_g), P(o_t))
    close(o_pe, pe, 1e-5, 2e-6, 'pe')
    close(o_g, xd.grad, 1e-4, 1e-4, 'pe backward')
    close(o_t, jt, 1e-4, 1e-4, 'pe tangent')
    x4 = torch.rand(50, 4, generator=g) * 2 - 1
    o4 = np.zeros((50, 84), np.float32)
    hc.hc_pe4(50, 10, P(f32(x4)), P(o4))
    close(o4, O.embed(x4.double(), 10), 1e-4, 1e-4, 'pe10')


def test_sdf_alpha(hc):
    g = torch.Generator().manual_seed(5)
    n = 500
    sdf = torch.randn(n, generator=g) * 0.05
    gr = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1) * (1 + 0.2 * torch.randn(n, 1, generator=g))
    dr = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    dist = torch.rand(n, generator=g) * 0.05 + 1e-3
    da, dge = torch.randn(n, generator=g), torch.randn(n, generator=g)
    for inv_s, car in [(20.0, 0.0), (80.0, 0.3), (300.0, 1.0)]:
        s, G = sdf.double().requires_grad_(True), gr.double().requires_grad_(True)
        iv = torch.tensor(inv_s, dtype=torch.float64, requires_grad=True)
        tc = (dr.double() * G).sum(-1)
        ic = -(torch.relu(-tc * 0.5 + 0.5) * (1 - car) + torch.relu(-tc) * car)
        pc = torch.sigmoid((s - ic * dist.double() * 0.5) * iv)
        nc = torch.sigmoid((s + ic * dist.double() * 0.5) * iv)
        alpha = ((pc - nc + 1e-5) / (pc + 1e-5)).clip(0, 1)
        ge = (torch.linalg.norm(G, dim=-1) - 1) ** 2
        ((alpha * da.double()).sum() + (ge * dge.double()).sum()).backward()
        oa, oge, ods, odg, odi = [np.zeros(s_, np.float32) for s_ in (n, n, n, (n, 3), n)]
        hc.hc_sdf_alpha(n, P(f32(sdf)), P(f32(gr)), P(f32(dr)), P(f32(dist)), ctypes.c_float(inv_s), ctypes.c_float(car), P(f32(da)),
                        P(f32(dge)), P(oa), P(oge), P(ods), P(odg), P(odi))
        close(oa, alpha, 1e-4, 1e-5, 'alpha')
        close(oge, ge, 1e-4, 1e-6, 'gerr')
        close(ods, s.grad, 2e-3, 2e-3, 'dsdf')
        close(odg, G.grad, 2e-3, 2e-3, 'dg')
        assert abs(odi.sum() - float(iv.grad)) < 2e-3 * (1 + abs(float(iv.grad)))


def test_geometry(hc):
    g = torch.Generator().manual_seed(6)
    n = 300
    G = torch.randn(n, 3, generator=g)
    V = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    dn, dr, dnov = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g), torch.randn(n, generator=g)
    Gd = G.double().requires_grad_(True)
    nn_ = torch.nn.functional.normalize(Gd, dim=-1)
    vv = V.double()
    nov = (nn_ * vv).sum(-1)
    r = nov[:, None] * nn_ * 2 - vv
    ((nn_ * dn.double()).sum() + (r * dr.double()).sum() + (nov * dnov.double()).sum()).backward()
    on, orr, onov, odg = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros((n, 3), np.float32)
    hc.hc_geometry(n, P(f32(G)), P(f32(V)), P(f32(dn)), P(f32(dr)), P(f32(dnov)), P(on), P(orr), P(onov), P(odg))
    close(on, nn_, 1e-5, 1e-6, 'n')
    close(orr, r, 1e-5, 2e-6, 'r')
    close(odg, Gd.grad, 1e-3, 1e-3, 'dg')


def test_sphere_direction(hc):
    """sphere_dir_fwd/bwd (math_shade.cuh) against offset_points_to_sphere + get_sphere_intersection + normalize
    (network/field.py:380-396, 560-563) and their fp64 autograd w.r.t. the direction; points inside, near and outside the
    0.999 sphere."""
    torch.manual_seed(11)
    n = 400
    p = torch.randn(n, 3)
    p = p / p.norm(dim=-1, keepdim=True) * torch.cat([torch.rand(n - 100) * 0.95, 0.99 + 0.03 * torch.rand(100)]).unsqueeze(-1)
    d = torch.nn.functional.normalize(torch.randn(n, 3), dim=-1)
    gs = torch.randn(n, 3)
    s_out, gd = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
    hc.hc_sphere_dir(n, P(f32(p)), P(f32(d)), P(f32(gs)), P(s_out), P(gd))
    sp = O.offset_points_to_sphere(p)
    close(s_out, torch.nn.functional.normalize(sp + d * O.get_sphere_intersection(sp, d), dim=-1), 2e-5, 2e-6, 'sphere direction')
    dd = d.double().requires_grad_(True)
    spd = O.offset_points_to_sphere(p.double())
    s64 = torch.nn.functional.normalize(spd + dd * O.get_sphere_intersection(spd, dd), dim=-1)
    (s64 * gs.double()).sum().backward()
    close(gd, dd.grad, 2e-4, 2e-5, 'd sphere direction / d dir')


def test_combine(hc):
    g = torch.Generator().manual_seed(7)
    n = 600
    lut = torch.from_numpy(np.fromfile(os.path.join(HERE, '..', 'assets', 'bsdf_256_256.bin'), dtype=np.float32).reshape(256, 256, 2).copy())
    x = torch.rand(n, 20, generator=g)
    x[:, 14] = torch.randn(n, generator=g) * 1.5          # inner weight (occ clamp both sides)
    x[:, 19] = torch.rand(n, generator=g) * 1.4 - 0.2     # NoV beyond [0,1]
    x[:, 5:14] *= 1.5
    dc = torch.randn(n, 3, generator=g)
    xd = x.double().requires_grad_(True)
    m, rough, alb = xd[:, 0:1], xd[:, 1:2], xd[:, 2:5]
    Ld, Ldir, Li, iw, Lh, wh, NoV = xd[:, 5:8], xd[:, 8:11], xd[:, 11:14], xd[:, 14:15], xd[:, 15:18], xd[:, 18:19], xd[:, 19:20]
    occ = torch.clamp(iw * 0.5 + 0.5, 0, 1)
    Ls = Li * occ + (Lh * torch.clamp(wh, 0, 1) + Ldir * (1 - torch.clamp(wh, 0, 1))) * (1 - occ)
    fg = O.fg_lookup(lut.double(), torch.cat([torch.clamp(NoV, 0, 1), torch.clamp(rough, 0, 1)], -1))
    color = torch.clamp(O.linear_to_srgb((1 - m) * alb * Ld + ((0.04 * (1 - m) + m * alb) * fg[:, 0:1] + fg[:, 1:2]) * Ls), 0, 1)
    (color * dc.double()).sum().backward()
    oc, od = np.zeros((n, 3), np.float32), np.zeros((n, 20), np.float32)
    hc.hc_combine(n, P(f32(x)), P(f32(lut)), P(f32(dc)), P(oc), P(od))
    close(oc, color, 1e-5, 2e-6, 'color')
    close(od, xd.grad, 2e-3, 2e-3, 'combine grads')


def test_nerf_post_and_srgb(hc):
    g = torch.Generator().manual_seed(8)
    n = 300
    dens = torch.randn(n, generator=g) * 5
    dens[:5] = 25.0
    dist = torch.rand(n, generator=g) * 0.5
    rgb = torch.randn(n, 3, generator=g) * 3
    da, dc = torch.randn(n, generator=g), torch.randn(n, 3, generator=g)
    D, Rg = dens.double().requires_grad_(True), rgb.double().requires_grad_(True)
    alpha = 1 - torch.exp(-torch.nn.functional.softplus(D) * dist.double())
    col = O.linear_to_srgb(torch.exp(torch.clamp(Rg, max=5.0)))
    ((alpha * da.double()).sum() + (col * dc.double()).sum()).backward()
    oa, oc, odd, odr = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros((n, 3), np.float32)
    hc.hc_nerf_post(n, P(f32(dens)), P(f32(dist)), P(f32(rgb)), P(f32(da)), P(f32(dc)), P(oa), P(oc), P(odd), P(odr))
    close(oa, alpha, 1e-5, 1e-6, 'nerf alpha')
    close(oc, col, 2e-5, 1e-5, 'nerf color')
    close(odd, D.grad, 1e-3, 1e-5, 'ddens')
    close(odr, Rg.grad, 1e-3, 1e-4, 'drgb')


def test_human(hc):
    g = torch.Generator().manual_seed(9)
    n = 400
    rays = O.synthetic_rays(n, seed=12)
    p = torch.randn(n, 3, generator=g) * 0.4
    r = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    rough = torch.rand(n, 1, generator=g)
    pose = rays['human_poses']
    dipe = torch.randn(n, 24, generator=g)
    rd, rg = r.double().requires_grad_(True), rough.double().requires_grad_(True)
    inter, dists, hits = O.get_camera_plane_intersection(p.double(), rd, pose.double())
    mean = inter[..., :2] * 0.3
    var = rg * (dists[:, None] * 0.3) ** 2
    hits = hits & (torch.norm(mean, dim=-1) < 1.5) & (dists > 0)
    hf = hits.double().unsqueeze(-1)
    enc = O.ipe(mean * hf, (var * hf).expand(n, 2), 0, 6)
    (enc * dipe.double()).sum().backward()
    oe, oh, odr, odg = np.zeros((n, 24), np.float32), np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
    hc.hc_human(n, P(f32(p)), P(f32(r)), P(f32(pose.reshape(n, 12))), P(f32(rough[:, 0])), P(f32(dipe)), P(oe), P(oh), P(odr), P(odg))
    assert (oh > 0).sum() > 20, 'too few human-light hits in the test inputs'
    np.testing.assert_array_equal(oh > 0, hits.numpy())
    close(oe, enc, 1e-3, 1e-4, 'ipe')
    close(odr, rd.grad, 5e-3, 5e-3, 'human dr')
    close(odg, rg.grad[:, 0], 5e-3, 5e-3, 'human drough')


@pytest.mark.parametrize('ggx', [0, 1])
def test_mc_sampling_and_brdf_weights(hc, ggx):
    """math_mc.cuh (stage II): sampled directions, D*G/(4 NoV p) and (1-HoV)^5 vs the oracle's shade_mixed terms, and their
    forward-mode d/d(roughness) vs the oracle's autograd in float64 (network/field.py:768-812, 932-975)."""
    import nero_oracle_mat as OM
    g = torch.Generator().manual_seed(9)
    n = 600
    nrm = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1)
    view = torch.nn.functional.normalize(nrm + 0.8 * torch.randn(n, 3, generator=g), dim=-1)
    a = 0.05 + 0.9 * torch.rand(n, 1, generator=g)
    az = torch.rand(n, generator=g)
    el = 0.06 + 0.94 * torch.rand(n, generator=g)
    spec = (torch.arange(n) % 3 != 0)
    fd, fs = 2.0 / 3.0, 1.0 / 3.0
    scfg = OM.shader_cfg({'geometry_type': 'ggx_smith' if ggx else 'schlick'})
    # oracle, one sample per point, float64, roughness requires grad
    N, V = nrm.double(), view.double()
    A = a.double().requires_grad_(True)
    refl = torch.sum(V * N, -1, keepdim=True) * N * 2 - V
    tab = torch.stack([az, el], -1).double()
    dd = torch.stack([OM.sample_diffuse_directions(tab[i:i + 1], N[i:i + 1])[0, 0] for i in range(n)])
    ds = torch.stack([OM.sample_specular_directions(tab[i:i + 1], refl[i:i + 1], A[i:i + 1])[0, 0] for i in range(n)])
    d = torch.where(spec[:, None], ds, dd)
    H = torch.nn.functional.normalize(V + d, dim=-1)
    HoV = OM.saturate_dot(H, V)
    NoH, NoL, NoV = OM.saturate_dot(N, H), OM.saturate_dot(N, d), OM.saturate_dot(N, V)
    D = OM.distribution_ggx(NoH, A)
    prob = torch.where(spec[:, None], D * NoH / (4 * HoV + 1e-5) * fs, NoL / np.pi * fd)
    w = D * OM.geometry_term(scfg, NoV, NoL, A) / (4 * NoV * prob + 1e-5)
    f5 = torch.clamp(1.0 - HoV, min=0.0, max=1.0) ** 5.0
    gw = torch.autograd.grad(w.sum(), A, retain_graph=True)[0][:, 0]
    gf = torch.autograd.grad(f5.sum(), A, retain_graph=True)[0][:, 0]
    gd = torch.stack([torch.autograd.grad(d[:, k].sum(), A, retain_graph=True)[0][:, 0] for k in range(3)], -1)
    o = {k: np.zeros(s_, np.float32) for k, s_ in dict(dir=(n, 3), w=n, f5=n, ddir=(n, 3), dw=n, df5=n).items()}
    hc.hc_mc(n, P(f32(nrm)), P(f32(view)), P(f32(a[:, 0])), P(f32(az)), P(f32(el)), P(np.ascontiguousarray(spec.numpy(), np.int32)), ggx,
             ctypes.c_float(fd), ctypes.c_float(fs), P(o['dir']), P(o['w']), P(o['f5']), P(o['ddir']), P(o['dw']), P(o['df5']))
    close(o['dir'], d, 1e-5, 2e-6, 'direction')
    close(o['ddir'], gd, 2e-4, 2e-5, 'd direction / d roughness')
    ok = (NoV[:, 0] > 0.05) & (w[:, 0].abs() < 1e4)           # away from the 1e-5-regularised singular corners
    wn, gwn = w[:, 0].detach().numpy(), gw.numpy()
    m = ok.numpy()
    close(o['w'][m], wn[m], 2e-4, 1e-5, 'specular weight')
    close(o['dw'][m], gwn[m], 2e-3, 2e-3 * np.abs(gwn[m]).mean(), 'd weight / d roughness')
    close(o['f5'], f5[:, 0], 2e-4, 1e-6, 'schlick factor')
    close(o['df5'], gf, 2e-3, 1e-5, 'd schlick / d roughness')
