"""Host logic of the weight EMA (algorithm.ema_decay): the decay schedule and the module / state_dict layout."""
import pytest
import torch

from opticalflowdiffusion_b200.config import compose
from opticalflowdiffusion_b200.optim import ema_weight


def _table(k, beta, after, every):
    """The schedule as a literal float64 table: copy up to ``after``, then every ``every`` steps the ema_pytorch warm-up
    (inv_gamma 1, power 2/3) capped at ``beta``."""
    if k <= after:
        return 1.0
    if (k - after) % every != 0:
        return None
    j = float(k - after)
    return 1.0 - min(beta, 1.0 - (1.0 + j) ** (-2.0 / 3.0))


@pytest.mark.parametrize("after,every", [(0, 1), (0, 7), (5, 3), (100, 10), (1, 1), (37, 1)])
@pytest.mark.parametrize("beta", [0.9999, 0.99, 0.5])
def test_ema_weight_schedule(after, every, beta):
    updates = 0
    for k in range(1, 501):
        got, want = ema_weight(k, beta, after, every), _table(k, beta, after, every)
        assert got == want, (k, got, want)
        updates += got is not None and k > after
    assert updates == (500 - after) // every
    # warm-up: the decay grows with j and reaches beta
    assert ema_weight(after + every, 0.999, after, every) == pytest.approx(1 - (1 - (1 + every) ** (-2 / 3)))
    assert ema_weight(after + 10 ** 6 * every, 0.999, after, every) == pytest.approx(1 - 0.999)


def _algo(target, *extra):
    from opticalflowdiffusion_b200 import FlowDiffuser
    torch.manual_seed(0)
    return FlowDiffuser(compose([f"algorithm.target={target}", *extra]).algorithm)


@pytest.mark.parametrize("target", ["flow", "joint", "target"])
def test_ema_unet_adds_exactly_its_keys(target):
    m = _algo(target, "algorithm.ema_decay=0.999")
    sd = m.state_dict()
    unet_keys = list(m.unet.state_dict())
    assert len(unet_keys) == 276 and len(sd) == 841 + 276
    assert [k for k in sd if k.startswith("ema_unet.")] == ["ema_unet." + k for k in unet_keys]
    assert set(sd) - {"ema_unet." + k for k in unet_keys} == set(_algo(target).state_dict())
    assert all(not p.requires_grad for p in m.ema_unet.parameters())
    online = {p.data_ptr() for p in m.model.parameters()}
    assert not online & {p.data_ptr() for p in m.ema_unet.parameters()}
    for k in unet_keys:                                   # starts as a copy, in its own storage
        assert torch.equal(sd["ema_unet." + k], sd["unet." + k]), k
    # the EMA sampler shares the schedule tables and follows the module
    assert m.ema_model.betas is m.model.betas and m.ema_model.model is not m.model.model
    m.double()
    assert m.ema_model.betas is m.model.betas and m.ema_model.betas.dtype == torch.float64
    assert m._diffusion(None) is m.ema_model and m._diffusion(False) is m.model


def test_ema_off_by_default():
    m = _algo("joint")
    assert m.cfg.ema_decay is None and m.ema_decay is None
    assert len(m.state_dict()) == 841 and not hasattr(m, "ema_unet")
    assert m._diffusion(None) is m.model
    with pytest.raises(ValueError):
        m._diffusion(True)


def test_ema_key_absent_from_config():
    from opticalflowdiffusion_b200 import FlowDiffuser
    cfg = compose(["algorithm.target=flow"]).algorithm
    del cfg["ema_decay"]
    with pytest.raises((AttributeError, KeyError)):
        cfg.ema_decay
    m = FlowDiffuser(cfg)
    assert len(m.state_dict()) == 841 and not hasattr(m, "ema_unet")


def test_checkpoint_rules_on_the_host():
    """load_checkpoint: EMA restored from an EMA checkpoint, initialised from the UNet when the checkpoint has none,
    ignored (and reported) by a model without EMA."""
    from opticalflowdiffusion_b200 import io_formats as IO
    src = _algo("flow", "algorithm.ema_decay=0.99", "algorithm.zero_init=false")
    with torch.no_grad():
        for p in src.ema_unet.parameters():
            p.add_(1.0)
    sd = {k: v.clone() for k, v in src.state_dict().items()}
    dst = _algo("flow", "algorithm.ema_decay=0.99")
    epoch = dst.ema_unet.weights_epoch
    assert IO.load_checkpoint(dst, {"state_dict": sd}) == {"missing": [], "unexpected": [], "ema_initialised": False}
    assert dst.ema_unet.weights_epoch == epoch + 1
    for k, v in dst.state_dict().items():
        assert torch.equal(v, sd[k]), k
    plain = {k: v for k, v in sd.items() if not k.startswith("ema_unet.")}
    dst = _algo("flow", "algorithm.ema_decay=0.99")
    assert IO.load_checkpoint(dst, {"state_dict": plain}) == {"missing": [], "unexpected": [], "ema_initialised": True}
    for (k, e), u in zip(dst.ema_unet.state_dict().items(), src.unet.state_dict().values()):
        assert torch.equal(e, u), k
    off = _algo("flow")
    rep = IO.load_checkpoint(off, {"state_dict": sd})
    assert rep["missing"] == [] and rep["unexpected"] == [] and sorted(rep["ignored"]) == sorted(
        k for k in sd if k.startswith("ema_unet."))
    assert torch.equal(off.unet.init_conv.weight, src.unet.init_conv.weight)
