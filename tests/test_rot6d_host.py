"""Host-side checks of the 126-D (rot6d) score network: weights recipe, argument errors, and the entry points that are
built for the 63-D axis network only.  No GPU needed: every check here fires before a device handle is made."""
import ctypes as C
import types

import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import fitting, likelihood, losses, prior, sampling, sde_lib, synthetic
from dposer_b200.model import ScoreModelFC


def rot6d_state_dict(seed, monkeypatch):
    """oracle.score_ref.make_state_dict with the pose width set to 126: the recipe reads POSE_D when it runs."""
    from oracle import score_ref
    monkeypatch.setattr(score_ref, 'POSE_D', 126)
    sd = score_ref.make_state_dict(seed)
    assert sd['pre_dense.weight'].shape == (1024, 126) and sd['post_dense.bias'].shape == (126,)
    return sd


@pytest.fixture(scope='module')
def model126():
    return synthetic.make_score_model(7, pose_dim=6)


@pytest.mark.parametrize('seed', [0, 42])
def test_rot6d_model_weights_match_oracle_recipe(seed, monkeypatch):
    m = synthetic.make_score_model(seed, pose_dim=6)
    assert m.pose_width == 126 and m.is_rot6d and m._geometry_ok
    ref = rot6d_state_dict(seed, monkeypatch)
    sd = m.state_dict()
    assert set(sd) == set(ref)
    for k in ref:
        assert torch.equal(sd[k], ref[k]), k
    assert sd['pre_dense.weight'].shape == (1024, 126) and sd['post_dense.weight'].shape == (126, 1024)


def test_plain_rot6d_constructor_matches_oracle_recipe(monkeypatch):
    """ScoreModelFC(cfg, 21, 6, 1024, 512, 2) under torch.manual_seed(s): every Linear equals the oracle recipe's (same
    registration order, same generator stream); GroupNorm affines are the default ones / zeros, which the recipe only
    randomises after all modules exist."""
    ref = rot6d_state_dict(5, monkeypatch)
    torch.manual_seed(5)
    sd = ScoreModelFC(synthetic.default_config(), 21, 6, 1024, 512, 2).state_dict()
    assert set(sd) == set(ref)
    for k in ref:
        if 'gnorm' in k:
            assert torch.equal(sd[k], torch.ones(1024) if k.endswith('weight') else torch.zeros(1024)), k
        else:
            assert torch.equal(sd[k], ref[k]), k


def test_other_widths_have_no_kernels():
    cfg = synthetic.default_config()
    assert not ScoreModelFC(cfg, 21, 4, 1024, 512, 2)._geometry_ok
    assert not ScoreModelFC(cfg, 21, 6, 512, 512, 2)._geometry_ok


@pytest.mark.parametrize('width', [63, 125, 127])
def test_forward_rejects_wrong_width(model126, width):
    with pytest.raises(ValueError, match='126'):
        model126(torch.zeros(4, width), torch.zeros(4))
    with pytest.raises(ValueError, match='126'):
        model126.raw_forward(torch.zeros(4, width), torch.zeros(1))


def test_forward_rejects_wrong_width_on_axis_model():
    m = synthetic.make_score_model(1)
    with pytest.raises(ValueError, match='63'):
        m(torch.zeros(2, 126), torch.zeros(2))


def test_sampler_rejects_shape_of_other_width(model126):
    cfg = synthetic.default_config()
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., 4), (8, 63), lambda x: x, 1e-3, device='cuda')
    with pytest.raises(ValueError, match='126'):
        fn(model126, z=torch.zeros(8, 63))


def test_likelihood_rejects_rot6d(model126):
    fn = likelihood.get_likelihood_fn(sde_lib.subVPSDE(0.1, 20., 1000), lambda x: x)
    with pytest.raises(NotImplementedError, match='rot6d'):
        fn(model126, torch.zeros(4, 126))


def test_device_rk45_ode_sampler_rejects_rot6d(model126):
    cfg = synthetic.default_config()
    cfg.sampling.method = 'ode'
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., 1000), (4, 126), lambda x: x, 1e-3, device='cuda')
    with pytest.raises(NotImplementedError, match='rot6d'):
        fn(model126, z=torch.zeros(4, 126))


def test_motion_denoise_rejects_rot6d(model126):
    args = types.SimpleNamespace(device=torch.device('cpu'))
    with pytest.raises(NotImplementedError, match='rot6d'):
        fitting.MotionDenoise(synthetic.default_config(), args, model126, None, sde_lib.subVPSDE(0.1, 20., 1000),
                              None, batch_size=4)


def test_smplify_rejects_rot6d_prior(model126):
    args = types.SimpleNamespace(device=torch.device('cpu'), sde_N=500, time_strategy='3')
    pose_prior = prior.DPoser(batch_size=1, args=args, model=model126, sde=sde_lib.subVPSDE(0.1, 20., 1000),
                              normalizer=object())
    with pytest.raises(NotImplementedError, match='rot6d'):
        fitting.SMPLify(None, batch_size=1, args=args, pose_prior=pose_prior)


def test_training_rejects_rot6d(model126):
    with pytest.raises(NotImplementedError, match='rot6d'):
        losses._Engine(model126, 8, torch.device('cpu'))


def test_c_abi_rejects_unsupported_widths():
    lib = L.load()
    out = C.c_void_p()
    w = L.ScoreWeights()
    for dim in (0, 64, 125, 128):
        assert lib.dpb_score_create_dim(C.byref(out), C.byref(w), dim, 0) == L.EUNSUPPORTED
        assert 'pose_dim' in lib.dpb_last_error().decode()
        assert lib.dpb_normal_fill_dim(None, 4, 0, 0, 1, dim, None) == L.EUNSUPPORTED
        assert lib.dpb_langevin_norms_dim(None, None, None, 4, dim, None) == L.EUNSUPPORTED
        assert lib.dpb_langevin_update_dim(None, None, None, None, None, 0.1, 0.1, 4, dim, None) == L.EUNSUPPORTED
    assert not out.value
    # a null weight struct with a supported width is an argument error, not a width error
    assert lib.dpb_score_create_dim(C.byref(out), None, 126, 0) == L.EINVAL
    assert lib.dpb_score_pose_dim(None) == L.EINVAL
    assert lib.dpb_normal_fill_dim(None, 4, 0, 0, 1, 126, None) == L.EINVAL


# Every public entry point that hands a pose tensor to a kernel indexes it as [B, D]: a tensor of the other width must be
# rejected before the handle is made (the models here live on the CPU, so reaching handle() would raise RuntimeError).
def _sde():
    return sde_lib.subVPSDE(0.1, 20., 1000)


def test_prior_losses_reject_wrong_width(model126):
    x63, x126 = torch.zeros(4, 63), torch.zeros(4, 126)
    comp = prior.DPoserComp(model126, _sde(), True, batch_size=4)
    mp = prior.MotionPrior(model126, _sde(), True, batch_size=4)
    args = types.SimpleNamespace(device=torch.device('cpu'), sde_N=1000)
    dp = prior.DPoser(batch_size=4, args=args, model=model126, sde=_sde(), normalizer=object())
    for multi in (False, True):
        with pytest.raises(ValueError, match='x_0'):
            comp.loss(x63, 0.5, multi_denoise=multi)
        with pytest.raises(ValueError, match='x_0'):
            mp.DPoser_loss(x63, 0.5, multi_denoise=multi)
        with pytest.raises(ValueError, match='x_0'):
            dp.DPoser_loss(x63, 0.5, multi_denoise=multi)
        with pytest.raises(ValueError, match='z'):
            comp.loss(x126, 0.5, multi_denoise=multi, z=x63)
        with pytest.raises(ValueError, match='z'):
            comp.loss(x126, 0.5, multi_denoise=multi, z=torch.zeros(3, 126))
    with pytest.raises(ValueError, match='x_t'):
        comp.multi_step_denoise(x63, 0.5, 0.05)


def test_completion_optimize_rejects_wrong_width(model126):
    comp = prior.DPoserComp(model126, _sde(), True, batch_size=4)
    with pytest.raises(ValueError, match='observation'):
        comp.optimize(torch.zeros(4, 63), torch.ones(4, 63), iterations=1, steps_per_iter=1)
    with pytest.raises(ValueError, match='mask'):
        comp.optimize(torch.zeros(4, 126), torch.ones(4, 63), iterations=1, steps_per_iter=1)
    with pytest.raises(ValueError, match='z_list'):
        comp.optimize(torch.zeros(4, 126), torch.ones(4, 126), iterations=1, steps_per_iter=1,
                      z_list=[torch.zeros(4, 63)])


def test_sampler_rejects_inputs_of_other_width(model126):
    cfg = synthetic.default_config()
    B, N = 8, 4
    fn = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, 126), lambda x: x, 1e-3, device='cuda')
    comp = types.SimpleNamespace(task='completion')
    ok = torch.zeros(B, 126)
    with pytest.raises(ValueError, match='z'):
        fn(model126, z=torch.zeros(B, 63))
    with pytest.raises(ValueError, match='observation'):
        fn(model126, z=ok, observation=torch.zeros(B, 63), mask=ok, args=comp)
    with pytest.raises(ValueError, match='mask'):
        fn(model126, z=ok, observation=ok, mask=torch.zeros(B, 63), args=comp)
    with pytest.raises(ValueError, match='observation'):
        fn(model126, z=ok, observation=torch.zeros(B - 1, 126), mask=ok, args=comp)
    for bad in (torch.zeros(N, 1, B, 63), torch.zeros(N - 1, 1, B, 126), torch.zeros(N, 1, B + 1, 126),
                torch.zeros(N, B, 126)):
        with pytest.raises(ValueError, match='noise'):
            fn(model126, z=ok, noise=bad)
    with pytest.raises(ValueError, match='noise'):                    # completion needs three planes per step
        fn(model126, z=ok, observation=ok, mask=ok, args=comp, noise=torch.zeros(N, 1, B, 126))
    cfg.sampling.corrector = 'langevin'
    fl = sampling.get_sampling_fn(cfg, sde_lib.subVPSDE(0.1, 20., N), (B, 126), lambda x: x, 1e-3, device='cuda')
    with pytest.raises(ValueError, match='noise'):                    # the Langevin draw comes first: two planes
        fl(model126, z=ok, noise=torch.zeros(N, 1, B, 126))
    with pytest.raises(ValueError, match='x'):
        sampling._run_steps(model126, torch.zeros(B, 63), None, None, None, None, None, 0, 0, None, None, False)
