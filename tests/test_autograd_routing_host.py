"""The routing rule every network's forward applies (models._EngineNet._differentiable / _dropout), on the host: which
calls take the differentiable path, and that an eval-mode differentiable call draws no dropout seed."""
import torch

from infodiffusion_b200.models import AuxiliaryUNet


def _net():
    return AuxiliaryUNet(T=10, ch=64, ch_mult=[1, 2], attn=[1], num_res_blocks=1, a_dim=8, shape=(3, 32, 32))


def test_differentiable_path_rule():
    net = _net().eval()
    x, a = torch.zeros(1, 3, 32, 32), torch.zeros(1, 8)
    assert net.head.weight.requires_grad
    assert not net._differentiable(x, a)                      # eval, inputs without grad: inference plan
    assert net._differentiable(x.clone().requires_grad_(), a)
    assert net._differentiable(x, a.clone().requires_grad_())
    assert not net._differentiable(x, None)
    with torch.no_grad():
        assert not net._differentiable(x.clone().requires_grad_(), a)
    net.train()
    assert net._differentiable(x, a)
    with torch.no_grad():
        assert not net._differentiable(x, a)


def test_dropout_seed_is_drawn_in_train_mode_only():
    net = _net()
    torch.manual_seed(3)
    state = torch.get_rng_state()
    assert net.eval()._dropout() == (0, 0.0)
    assert torch.equal(torch.get_rng_state(), state)
    seed, p = net.train()._dropout()
    assert p == net.dropout_p > 0
    assert not torch.equal(torch.get_rng_state(), state)
    torch.manual_seed(3)
    assert net._dropout()[0] == seed                          # follows torch.manual_seed
