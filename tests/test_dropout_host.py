"""CPU: host side of native ResBlock dropout — the engine's dropout probability, and the argument checks of the dropout fields of
fdm_gn_apply / fdm_gn_bwd (they return before any CUDA call)."""
import ctypes
import math

import pytest

PIXEL = dict(diffusion_space="pixel", pre_encoded=False, pre_encoded_stats_dict=None)


def _model(dropout):
    from improved_diffusion.script_util import create_model_and_diffusion, model_and_diffusion_defaults
    d = model_and_diffusion_defaults()
    d.update(image_size=32, in_channels=4, num_channels=32, num_res_blocks=1, diffusion_steps=32, dropout=dropout,
             diffusion_space_kwargs=dict(PIXEL))
    return create_model_and_diffusion(**d)[0]


def test_train_dropout_follows_the_mode():
    """The engine's dropout probability is the model's `dropout` in train mode and 0 in eval mode, as nn.Dropout behaves; a value
    outside [0, 1] is refused.  (That native training on CPU tensors refuses dropout loudly is checked in test_host_cpu.py.)"""
    model = _model(0.1)
    eng = model.engine()
    for train, p in ((True, 0.1), (False, 0.0)):
        model.train(train)
        assert eng.train_dropout() == p
    model.train()
    model.dropout = 1.5
    with pytest.raises(ValueError, match="dropout"):
        eng.train_dropout()


def _fake(n):
    return ctypes.c_void_p(0x1000 * n)  # never dereferenced: the calls below return at argument validation


@pytest.mark.parametrize("p,silu", [(-0.1, 1), (1.5, 1), (math.nan, 1), (0.1, 0)])
def test_dropout_arguments_are_validated(p, silu):
    """drop_p outside [0, 1] (NaN included), or dropout on a launch without SiLU: FDM_ERR_BAD_ARG."""
    from improved_diffusion import _native as N_
    L = N_.lib()
    philox = _fake(9)
    ga = N_.GnApplyArgs(xa=_fake(1), stats_a=_fake(2), gamma=_fake(3), beta=_fake(4), out_op=_fake(5), N=1, HW=16, Ca=32, T=1,
                        silu=silu, eps=1e-5, drop_philox=philox, drop_p=p, drop_salt=1)
    assert L.fdm_gn_apply(ctypes.byref(ga), None) == -1
    gb = N_.GnBwdArgs(xa=_fake(1), stats_a=_fake(2), gamma=_fake(3), beta=_fake(4), dy_op=_fake(5), gxa=_fake(6), ab=_fake(7),
                      dgamma=_fake(8), dbeta=_fake(10), N=1, HW=16, Ca=32, T=1, silu=silu, eps=1e-5, drop_philox=philox, drop_p=p,
                      drop_salt=1)
    assert L.fdm_gn_bwd(ctypes.byref(gb), None) == -1
