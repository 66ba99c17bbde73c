"""Pins the oracle (oracle/*.py) against golden vectors produced by the unmodified reference
(tests/golden/gen_golden.py).  CPU only."""
import os
import numpy as np
import torch

import unet_oracle as UO
import deblur_oracle as DO

G = os.path.join(os.path.dirname(__file__), 'golden')


def load(name):
    z = np.load(os.path.join(G, name + '.npz'))
    return {k: torch.from_numpy(np.asarray(z[k])) for k in z.files}


def rel(a, b):
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def test_unet_forward_loss_grads_match_reference():
    g = load('unet_small')
    sd = {k[3:]: v.clone().requires_grad_(True) for k, v in g.items() if k.startswith('sd:')}
    y = UO.unet_forward(sd, g['x'], g['t'])
    assert rel(y.detach(), g['y']) < 2e-6
    loss = (g['target'] - y).abs().mean()
    assert abs(loss.item() - g['loss'].item()) < 1e-6
    loss.backward()
    n = 0
    for k, v in g.items():
        if k.startswith('grad:'):
            assert rel(sd[k[5:]].grad, v) < 2e-5, k
            n += 1
        elif k.startswith('gsub:'):
            gr = sd[k[5:]].grad.reshape(-1)
            stride = gr.numel() // 2048
            assert rel(gr[::stride], v) < 2e-5, k
            assert abs(gr.double().norm().item() / g['gnorm:' + k[5:]].item() - 1) < 1e-5
            n += 1
    assert n == len(sd)


def test_make_state_dict_has_reference_keys_and_shapes():
    g = load('unet_small')
    ref = {k[3:]: tuple(v.shape) for k, v in g.items() if k.startswith('sd:')}
    mine = {k: tuple(v.shape) for k, v in UO.make_unet_state_dict(32, (1, 2), 3).items()}
    assert ref == mine


def _cases(prefix, g):
    return sorted(k[len(prefix):] for k in g if k.startswith(prefix))


def test_blur_weights_and_q_sample_match_reference():
    g = load('qsample')
    x = g['x']
    for key in _cases('q:', g):
        routine, ks, std, T, disc = key.split('|')
        o = DO.DeblurOracle(None, image_size=16, channels=3, timesteps=int(T), kernel_std=float(std),
                            kernel_size=int(ks), blur_routine=routine, discrete=bool(int(disc)))
        w = torch.stack(o.kernels2d)
        assert torch.equal(w, g['w:' + key]), key          # taps bit-exact vs reference+shim
        q = o.q_sample(x, g['t:' + key])
        if int(disc):
            # 8-bit truncation can flip one level on a last-ulp difference; allow <=1 level on <0.1% of pixels
            d = (q - g['q:' + key]).abs()
            assert d.max() <= 2 / 255 + 1e-6 and (d > 1e-6).float().mean() < 1e-3, key
        else:
            assert torch.allclose(q, g['q:' + key], atol=2e-6, rtol=0), key


def test_sample_and_p_losses_match_reference():
    g = load('sample_small')
    u = load('unet_small')
    sd = {k[3:]: v for k, v in u.items() if k.startswith('sd:')}
    fn = lambda x, t: UO.unet_forward(sd, x, t)
    for key in _cases('img:', g):
        routine, ks, std, T, samp, disc = key.split('|')
        o = DO.DeblurOracle(fn, image_size=32, channels=3, timesteps=int(T), kernel_std=float(std),
                            kernel_size=int(ks), blur_routine=routine, sampling_routine=samp,
                            discrete=bool(int(disc)))
        xt, dr, img = o.sample(2, g['x'])
        assert rel(xt, g['xt:' + key]) < 1e-5, key
        assert rel(dr, g['dr:' + key]) < 1e-5, key
        assert rel(img, g['img:' + key]) < 1e-4, key
        with torch.no_grad():
            loss = o.p_losses(g['x'], torch.tensor([int(T) - 1, 0]))
        assert abs(loss.item() - g['loss:' + key].item()) < (2e-3 if int(disc) else 1e-5), key


def test_denoise_oracle_matches_reference():
    import denoise_oracle as NO
    g = load('denoise_small')
    u = load('unet_small')
    sd = {k[3:]: v for k, v in u.items() if k.startswith('sd:')}
    fn = lambda x, t: UO.unet_forward(sd, x, t)
    for samp in ('ddim', 'x0_step_down'):
        o = NO.DenoiseOracle(fn, image_size=32, timesteps=5, sampling_routine=samp)
        assert torch.allclose(o.sa, g['sqrt_ac'], atol=1e-7) and torch.allclose(o.sb, g['sqrt_1mac'], atol=1e-7)
        tt = torch.tensor([4, 0])
        assert torch.allclose(o.q_sample(g['x1'], g['x2'], tt), g['q:' + samp], atol=1e-6)
        with torch.no_grad():
            assert abs(o.p_losses(g['x1'], g['x2'], tt).item() - g['loss:' + samp].item()) < 1e-5
        _, dr, img = o.gen_sample(2, g['x2'])
        assert rel(dr, g['dr:' + samp]) < 1e-5 and rel(img, g['img:' + samp]) < 1e-4
    o = NO.DenoiseOracle(fn, image_size=32, timesteps=5)
    _, dr, img = o.sample(2, g['x2'])
    assert rel(dr, g['sample_dr']) < 1e-5 and rel(img, g['sample_img']) < 1e-4


def test_resolution_oracle_matches_reference():
    import resolution_oracle as RO
    g = load('resolution_small')
    u = load('unet_small')
    sd = {k[3:]: v for k, v in u.items() if k.startswith('sd:')}
    fn = lambda x, t: UO.unet_forward(sd, x, t)
    for key in _cases('img:', g):
        routine, T, samp = key.split('|')
        o = RO.ResolutionOracle(fn, image_size=32, timesteps=int(T), resolution_routine=routine, sampling_routine=samp)
        tt = torch.tensor([int(T) - 1, 1])
        assert torch.allclose(o.q_sample(g['x'], tt), g['q:' + key], atol=1e-6), key
        with torch.no_grad():
            assert abs(o.p_losses(g['x'], tt).item() - g['loss:' + key].item()) < 1e-5
        xt, dr, img = o.sample(2, g['x'])
        assert rel(xt, g['xt:' + key]) < 1e-6 and rel(dr, g['dr:' + key]) < 1e-5 and rel(img, g['img:' + key]) < 1e-4, key


def test_defading_oracle_matches_reference():
    import defading_oracle as FO
    g = load('defading_small')
    u = load('unet_small')
    sd = {k[3:]: v for k, v in u.items() if k.startswith('sd:')}
    fn = lambda x, t: UO.unet_forward(sd, x, t)
    for key in _cases('img:', g):
        routine, T, samp, disc = key.split('|')
        o = FO.DefadeOracle(fn, image_size=32, timesteps=int(T), kernel_std=0.6, initial_mask=3, fade_routine=routine,
                            sampling_routine=samp, discrete=bool(int(disc)))
        assert torch.equal(o.fade_kernels, g['k:' + key]), key            # masks bit-exact
        rx, ry = (g['rx:' + key], g['ry:' + key]) if 'Random' in routine else (None, None)
        tt = torch.tensor([int(T) - 1, 0])
        q = o.q_sample(g['x'], tt, rx, ry)
        if int(disc):
            assert (q - g['q:' + key]).abs().max() <= 2 / 255 + 1e-6
        else:
            assert torch.allclose(q, g['q:' + key], atol=1e-6), key
        xt, dr, img = o.sample(2, g['x'], rx=rx, ry=ry)
        tol = 5e-3 if int(disc) else 1e-4
        assert rel(xt, g['xt:' + key]) < tol and rel(dr, g['dr:' + key]) < tol and rel(img, g['img:' + key]) < max(tol, 1e-4), key


def _snow_cfg(key):
    fpt, kws, T, samp = key.split('|')
    kw = {}
    for item in kws.split('-'):
        k, v = item.split('=')
        kw[k] = (v == 'True') if v in ('True', 'False') else (float(v) if '.' in v else (int(v) if v.isdigit() else v))
    return fpt, kw, int(T), samp


def test_snow_decolor_oracle_and_host_tables_match_reference():
    import snow_oracle as SO
    from cold_diffusion_models_b200.snowification import DeColorization
    g = load('snow_small')
    u = load('unet_small')
    sd = {k[3:]: v for k, v in u.items() if k.startswith('sd:')}
    fn = lambda x, t: UO.unet_forward(sd, x, t)
    for key in _cases('img:', g):
        fpt, kw, T, samp = _snow_cfg(key)
        if fpt == 'Decolorization':
            host = DeColorization(num_timesteps=T, **kw)
            fp = SO.DecolorFP(host.factors)
        else:
            layers, br = SO.generate_snow_layers((32, 32), snow_level=kw.get('snow_level', 1), num_timesteps=T)
            assert torch.allclose(layers, g['snow:' + key], atol=1e-6), key     # oracle snow-layer generator == reference layers
            assert torch.allclose(torch.tensor(br), g['br:' + key], atol=1e-7)
            fp = SO.SnowFP(layers, br, fix_brightness=kw.get('fix_brightness', False))
        o = SO.SnowOracle(fn, fp, timesteps=T, sampling_routine=samp)
        assert torch.allclose(o.q_sample(g['x'], torch.tensor([T - 1, -1, 1])), g['q:' + key], atol=2e-6), key
        with torch.no_grad():
            assert abs(o.p_losses(g['x'], torch.tensor([T - 1, 0, 1])).item() - g['loss:' + key].item()) < 1e-5
        x1, d1 = o.sample_one_step(g['x'], torch.tensor([T - 1, 1, 2]))
        assert rel(x1, g['one_x:' + key]) < 1e-5 and rel(d1, g['one_dr:' + key]) < 1e-5, key
        r = o.sample(3, g['x'])
        assert rel(r['xt'], g['xt:' + key]) < 1e-6 and rel(r['direct_recons'], g['dr:' + key]) < 1e-5 and rel(r['recon'], g['img:' + key]) < 1e-4, key


def test_model2_oracle_matches_reference():
    import model2_oracle as MO
    g = load('model2_small')
    sd = {k[3:]: v for k, v in g.items() if k.startswith('sd:')}
    with torch.no_grad():
        y = MO.model_forward(sd, g['x'], g['t'], ch=32, num_resolutions=2, num_res_blocks=2)
    assert rel(y, g['y']) < 2e-6
    fn = lambda x, t: MO.model_forward(sd, x, t, ch=32, num_resolutions=2, num_res_blocks=2)
    o = DO.DeblurOracle(fn, image_size=16, channels=3, timesteps=6, kernel_std=0.1, kernel_size=3, blur_routine='Special_6_routine',
                        sampling_routine='x0_step_down')
    xt, dr, img = o.sample(3, g['x'])
    assert rel(xt, g['s_xt']) < 1e-5 and rel(dr, g['s_dr']) < 1e-5 and rel(img, g['s_img']) < 1e-4


def test_oracle_matches_reference_config1_mnist():
    """BASELINE config 1: MNIST-shaped 1x32x32, T=20, k=11, sigma=7, Constant, B=4, full-size Unet, against the reference's
    loss and network output (tests/golden/gen_golden_config1.py; the weights are rebuilt from their seed)."""
    g = load('config1_mnist')
    sd = UO.make_unet_state_dict(64, (1, 2, 4, 8), 1, seed=0)
    o = DO.DeblurOracle(lambda a, b: UO.unet_forward(sd, a, b), image_size=32, channels=1, timesteps=20,
                        kernel_std=7.0, kernel_size=11, blur_routine='Constant')
    x, t = g['x'], g['t']
    with torch.no_grad():
        loss = o.p_losses(x, t)
        y = UO.unet_forward(sd, o.q_sample(x, t), t)
    assert abs(loss.item() - g['loss'].item()) < 1e-5
    assert rel(y, g['y']) < 1e-5


def _small_fn():
    u = load('unet_small')
    sd = {k[3:]: v for k, v in u.items() if k.startswith('sd:')}
    return lambda x, t: UO.unet_forward(sd, x, t)


def test_demixing_oracle_matches_reference():
    import demixing_oracle as MO
    g = load('demixing_small')
    o = MO.DemixingOracle(_small_fn(), image_size=32, timesteps=5)
    x1, x2, tt = g['x1'], g['x2'], torch.tensor([4, 1])
    assert torch.allclose(o.q_sample(x1, x2, tt), g['q'], atol=1e-6)
    with torch.no_grad():
        assert abs(o.p_losses(x1, x2, tt).item() - g['loss'].item()) < 1e-5
    _, dr, img = o.gen_sample(2, x2)
    assert rel(dr, g['gen_dr']) < 1e-5 and rel(img, g['gen_img']) < 1e-4
    _, dr, img = o.sample(2, x2)
    assert rel(dr, g['sample_dr']) < 1e-5 and rel(img, g['sample_img']) < 1e-4
    F_, B_, img = o.forward_and_backward(2, x1, x2)
    assert rel(torch.stack(F_), g['fb_F']) < 1e-6 and rel(torch.stack(B_), g['fb_B']) < 1e-4 and rel(img, g['fb_img']) < 1e-4
    X1, Xt = o.all_sample(2, x2)
    assert rel(torch.stack(X1), g['all_X1']) < 1e-4 and rel(torch.stack(Xt), g['all_Xt']) < 1e-4


def test_defading_generation_oracle_matches_reference():
    import defading_gen_oracle as GO
    g = load('defading_gen_small')
    fn = _small_fn()
    x1, col, tt = g['x1'], g['col'], torch.tensor([3, 0])
    for rev in (False, True):
        k = 'rev%d:' % int(rev)
        o = GO.DefadingGenOracle(fn, image_size=32, timesteps=4, reverse=rev, kernel_std=0.6, initial_mask=3)
        assert torch.allclose(o.alphas, g[k + 'alphas'], atol=1e-6) and torch.allclose(o.one_minus_alphas, g[k + 'one_minus_alphas'], atol=1e-6)
        assert torch.allclose(o.q_sample(x1, col, tt), g[k + 'q'], atol=2e-6)
        with torch.no_grad():
            assert abs(o.p_losses(x1, col, tt).item() - g[k + 'loss'].item()) < 1e-5
        _, dr, img = o.sample(2, col)
        assert rel(dr, g[k + 'sample_dr']) < 1e-5 and rel(img, g[k + 'sample_img']) < 1e-4
        _, dr, img = o.gen_sample(2, col)
        assert rel(dr, g[k + 'gen_dr']) < 1e-5 and rel(img, g[k + 'gen_img']) < 1e-4
        F_, B_, img = o.forward_and_backward(2, x1, col)
        assert rel(torch.stack(F_), g[k + 'fb_F']) < 1e-5 and rel(torch.stack(B_), g[k + 'fb_B']) < 1e-4 and rel(img, g[k + 'fb_img']) < 1e-4
        X1, Xt = o.all_sample(2, col)
        assert rel(torch.stack(X1), g[k + 'all_X1']) < 1e-4 and rel(torch.stack(Xt), g[k + 'all_Xt']) < 1e-4


def test_deblur_cover_trajectories_match_reference():
    g = load('fb_small')
    fn = _small_fn()
    x = g['x']
    for key in _cases('img:', g):
        routine, ks, std, T, samp = key.split('|')
        o = DO.DeblurOracle(fn, image_size=32, channels=3, timesteps=int(T), kernel_std=float(std), kernel_size=int(ks),
                            blur_routine=routine, sampling_routine=samp)
        F_, B_, img = o.forward_and_backward(2, x)
        assert rel(torch.stack(F_), g['F:' + key]) < 1e-5 and rel(torch.stack(B_), g['B:' + key]) < 1e-4, key
        assert rel(img, g['img:' + key]) < 1e-4, key
        F2, B1, B2, i1, i2 = o.forward_and_backward_2(2, x)
        assert rel(torch.stack(F2), g['F2:' + key]) < 1e-5, key
        assert rel(torch.stack(B1), g['B1:' + key]) < 1e-4 and rel(torch.stack(B2), g['B2:' + key]) < 1e-4, key
        assert rel(i1, g['i1:' + key]) < 1e-4 and rel(i2, g['i2:' + key]) < 1e-4, key


def test_model2_oracle_gradients_match_reference():
    """autograd through the functional restatement of Model2.py reproduces every parameter gradient of the reference `Model`
    (L1 loss, dropout inactive) -- the checker for the Model training path."""
    import model2_oracle as MO
    g = load('model2_small')
    gg = load('model2_grads_small')
    sd = {k[3:]: v.clone().requires_grad_(v.dtype.is_floating_point) for k, v in g.items() if k.startswith('sd:')}
    y = MO.model_forward(sd, g['x'], g['t'], ch=32, num_resolutions=2, num_res_blocks=2)
    loss = (gg['target'] - y).abs().mean()
    assert abs(loss.item() - gg['loss'].item()) < 1e-6
    loss.backward()
    n = 0
    for k, v in gg.items():
        if k.startswith('grad:'):
            if v.abs().max() < 1e-7:
                # zero in exact arithmetic (a per-channel shift in front of a one-channel GroupNorm group: conv1.bias / temb_proj
                # at ch = 32; the key bias in front of a row softmax): round-off on both sides, whose pattern changes with the
                # number of CPU threads, so the check is absolute, as in tests/test_model2_host_logic.py
                assert sd[k[5:]].grad.abs().max() < 1e-7, k
            else:
                assert rel(sd[k[5:]].grad, v) < 3e-5, k
            n += 1
        elif k.startswith('gsub:'):
            gr = sd[k[5:]].grad.reshape(-1)
            stride = gr.numel() // 2048
            assert rel(gr[::stride], v) < 3e-5, k
            assert abs(gr.double().norm().item() / gg['gnorm:' + k[5:]].item() - 1) < 1e-5, k
            n += 1
    assert n == sum(1 for v in sd.values() if v.requires_grad)


def test_individual_incremental_routine_matches_reference():
    """the seventh blur routine: kernel size 2i+1, sigma 2k, single-kernel head in `sample` (DB:379-383, 401-402, 429-430)"""
    g = load('individual_small')
    fn = _small_fn()
    x = g['x']
    for samp in ('default', 'x0_step_down'):
        o = DO.DeblurOracle(fn, image_size=32, channels=3, timesteps=4, kernel_std=0.1, kernel_size=3,
                            blur_routine='Individual_Incremental', sampling_routine=samp)
        for i, w in enumerate(o.kernels2d):
            assert torch.equal(w, g['w%d' % i])
        tt = torch.tensor([3, 1])
        assert torch.allclose(o.q_sample(x, tt), g['q'], atol=2e-6)
        with torch.no_grad():
            assert abs(o.p_losses(x, tt).item() - g['loss'].item()) < 1e-5
        xt, dr, img = o.sample(2, x)
        assert rel(xt, g['xt:' + samp]) < 1e-5 and rel(dr, g['dr:' + samp]) < 1e-5 and rel(img, g['img:' + samp]) < 1e-4, samp


def test_resolution_train_routines_match_reference():
    """the research train routines of the resolution package (RS:655-761) and the t = -1 quirk of its q_sample (RS:645)"""
    import resolution_oracle as RO
    g = load('resolution_train_small')
    fn = _small_fn()
    x, tt = g['x'], torch.tensor([3, 0, 2])
    for key in _cases('loss:', g):
        routine, lt = key.split('|')
        o = RO.ResolutionOracle(fn, image_size=32, timesteps=4, resolution_routine='Incremental_factor_2', sampling_routine='x0_step_down',
                                loss_type=lt)
        torch.manual_seed(7)
        with torch.no_grad():
            assert abs(float(o.p_losses(x, tt, train_routine=routine)) - g['loss:' + key].item()) < 1e-5, key
    assert torch.allclose(o.q_sample(x, torch.tensor([2, -1, 1])), g['q_neg'], atol=1e-6)
