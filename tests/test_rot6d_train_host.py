"""Host-side checks of training, likelihood and the probability-flow ODE for 126-D (rot6d) score networks: width errors
of the C ABI and of the Python entry points, all raised before any device is touched (no GPU needed)."""
import ctypes as C
import types

import pytest
import torch

from dposer_b200 import _lib as L
from dposer_b200 import likelihood, losses, ode, sampling, sde_lib, synthetic


@pytest.fixture(scope='module')
def model126():
    return synthetic.make_score_model(7, pose_dim=6)


@pytest.fixture(scope='module')
def model63():
    return synthetic.make_score_model(7)


def _sde():
    return sde_lib.subVPSDE(0.1, 20., 1000)


def test_c_abi_rejects_unsupported_widths():
    lib = L.load()
    out = C.c_void_p()
    for dim in (0, 64, 125, 128):
        assert lib.dpb_train_create_dim(C.byref(out), 8, dim, 0) == L.EUNSUPPORTED
        assert 'pose_dim' in lib.dpb_last_error().decode()
        assert lib.dpb_pf_ode_rhs_dim(None, None, None, None, 0.0, 0.0, None, 4, dim, None) == L.EUNSUPPORTED
        assert 'pose_dim' in lib.dpb_last_error().decode()
    assert not out.value
    # a supported width with bad arguments is an argument error, not a width error
    assert lib.dpb_train_create_dim(None, 8, 126, 0) == L.EINVAL
    assert lib.dpb_train_create_dim(C.byref(out), 0, 126, 0) == L.EINVAL
    assert lib.dpb_pf_ode_rhs_dim(None, None, None, None, 0.0, 0.0, None, 4, 126, None) == L.EINVAL


def test_jvp_workspace_of_a_null_handle_is_zero():
    lib = L.load()
    assert lib.dpb_score_jvp_workspace_bytes(None, 16) == 0


@pytest.mark.parametrize('width', [63, 125, 127])
def test_training_batches_of_the_other_width_are_value_errors(model126, width):
    sde = _sde()
    rows = torch.zeros(6, 4)
    with pytest.raises(ValueError, match='126'):
        losses.native_loss(model126, torch.zeros(4, width), rows)
    for fn in (losses.get_sde_loss_fn(sde, True, reduce_mean=True),
               losses.get_ddpm_loss_fn(sde_lib.VPSDE(0.1, 20., 1000), True),
               losses.get_smld_loss_fn(sde_lib.VESDE(0.01, 50., 1000), True)):
        with pytest.raises(ValueError, match=f'126.*{width}'):
            fn(model126, torch.zeros(4, width))
    with pytest.raises(ValueError, match='z'):
        losses.native_loss(model126, torch.zeros(4, 126), rows, z=torch.zeros(4, width))


def test_axis_network_rejects_rot6d_batches(model63):
    with pytest.raises(ValueError, match='63.*126'):
        losses.native_loss(model63, torch.zeros(4, 126), torch.zeros(6, 4))


def test_step_fn_rejects_batches_of_the_other_width(model126):
    cfg = synthetic.default_config()
    state = dict(model=model126, optimizer=types.SimpleNamespace(zero_grad=lambda: None), ema=None, step=0)
    for graph in (False, True):
        step_fn = losses.get_step_fn(_sde(), train=True, optimize_fn=losses.optimization_manager(cfg), graph=graph)
        with pytest.raises(ValueError, match='126'):
            step_fn(state, torch.zeros(4, 63))


def test_loss_reduction_follows_the_network_width(model63, model126):
    """reduce_mean's 1 / D is read from the model the loss function is called with, not fixed when it is built."""
    fn = losses.get_sde_loss_fn(_sde(), True, reduce_mean=True)
    t = torch.full((3,), 0.5)
    assert torch.allclose(fn.make_rows(model63, 3, t)[5], torch.full((3,), 1 / 63))
    assert torch.allclose(fn.make_rows(model126, 3, t)[5], torch.full((3,), 1 / 126))
    ddpm = losses.get_ddpm_loss_fn(sde_lib.VPSDE(0.1, 20., 1000), True, reduce_mean=True)
    assert torch.allclose(ddpm.make_rows(model126, 3, torch.tensor([1, 2, 3]))[5], torch.full((3,), 1 / 126))
    summed = losses.get_sde_loss_fn(_sde(), True, reduce_mean=False)
    assert torch.allclose(summed.make_rows(model126, 3, t)[5], torch.full((3,), 0.5))


def test_auxiliary_loss_rejects_rot6d(model126):
    with pytest.raises(NotImplementedError, match='rot6d'):
        losses.auxiliary_loss_grad(model126, _sde(), torch.zeros(4, 126), None, None)
    cfg = synthetic.default_config()
    step_fn = losses.get_step_fn(_sde(), train=True, optimize_fn=losses.optimization_manager(cfg), auxiliary_loss=True,
                                 denormalize=lambda v: v, body_model=object(), rot_rep='axis')
    with pytest.raises(NotImplementedError, match='rot6d'):
        step_fn(dict(model=model126, optimizer=None, ema=None, step=0), torch.zeros(4, 126))


def test_rot6d_training_engine_needs_cuda(model126):
    with pytest.raises(NotImplementedError, match='no CPU implementation'):
        losses._Engine(model126, 8, torch.device('cpu'))


def test_likelihood_rejects_data_of_the_other_width(model126, model63):
    fn = likelihood.get_likelihood_fn(_sde(), lambda x: x)
    with pytest.raises(ValueError, match='data'):
        fn(model126, torch.zeros(4, 63))
    with pytest.raises(ValueError, match='epsilon'):
        fn(model126, torch.zeros(4, 126), epsilon=torch.zeros(4, 63))
    with pytest.raises(ValueError, match='data'):
        fn(model63, torch.zeros(4, 126))
    with pytest.raises(NotImplementedError, match='no CPU implementation'):
        fn(model126, torch.zeros(4, 126))
    for method in ('RK23', 'RK45'):
        with pytest.raises(ValueError, match='data'):
            likelihood.get_likelihood_fn(_sde(), lambda x: x, method=method)(model126, torch.zeros(4, 63))


def test_ode_sampler_rejects_shapes_and_z_of_the_other_width(model126):
    cfg = synthetic.default_config()
    cfg.sampling.method = 'ode'
    fn = sampling.get_sampling_fn(cfg, _sde(), (4, 126), lambda x: x, 1e-3, device='cuda')
    with pytest.raises(ValueError, match='z'):
        fn(model126, z=torch.zeros(4, 63))
    bad = sampling.get_sampling_fn(cfg, _sde(), (4, 63), lambda x: x, 1e-3, device='cuda')
    with pytest.raises(ValueError, match='126'):
        bad(model126)
    host = sampling.get_ode_sampler(_sde(), (4, 126), lambda x: x, method='RK23', device='cpu')
    with pytest.raises(NotImplementedError, match='no CPU implementation'):
        host(model126, z=torch.zeros(4, 126))


def test_pf_ode_backend_rejects_the_other_width(model126):
    with pytest.raises(ValueError, match='x'):
        ode.PFOdeBackend(model126, _sde(), torch.zeros(4, 63))
    with pytest.raises(ValueError, match='epsilon'):
        ode.PFOdeBackend(model126, _sde(), torch.zeros(4, 126), torch.zeros(4, 63))
    with pytest.raises(ValueError, match='epsilon'):
        likelihood.drift_and_div(model126, _sde(), torch.zeros(4, 126), 0.5, torch.zeros(3, 126))
