"""The op plan + backward schedule, executed kernel-contract by kernel-contract on the CPU (plan emulator),
must reproduce the oracle's outputs, loss and every parameter gradient."""
import pytest
import torch

from oracle import cunet_oracle
from tests import plan_emulator
from cunet_b200 import plan as plan_mod


@pytest.mark.parametrize("cfg", [(5, 2, 1, 2), (4, 3, 2, 2), (3, 3, 0, 3), (6, 4, 1, 2), (3, 4, 3, 4)],
                         ids=["L2K1", "L3K2", "L3K0", "L4K1", "L4K3"])
def test_plan_matches_oracle(cfg):
    class_num, L, K, loss_num = cfg
    plan = plan_mod.Plan(class_num, L, K, loss_num, in_res=64)
    state = cunet_oracle.init_state(class_num, L, K, seed=3)
    gen = torch.Generator().manual_seed(7)
    # 4 images: with 2, the BatchNorms of the 1x1 neck normalise over two values, and that ill-conditioning amplifies
    # float64 rounding into ~1e-4 gradient differences that depend on the host CPU's summation order
    img = torch.rand(4, 3, 64, 64, generator=gen)
    hm = torch.rand(4, class_num, 16, 16, generator=gen)
    net = cunet_oracle.OracleCUNet({k: v.double() if v.is_floating_point() else v for k, v in state.items()},
                                   class_num, L, K, loss_num)
    for n in net.param_names:
        net.state[n] = net.state[n].detach().double().requires_grad_(True)
    outs = net(img.double())
    loss = cunet_oracle.multi_loss_mse(outs, hm.double())
    loss.backward()
    heads, eloss, grads = plan_emulator.run(plan, state, img, hm)
    assert abs(float(eloss) - float(loss.detach())) < 1e-7 * max(1.0, abs(float(loss)))
    for a, b in zip(heads, outs):
        assert (a - b.detach()).abs().max() < 1e-6
    used = 0
    for n in net.param_names:
        g = net.state[n].grad
        if g is None:
            assert n not in grads or grads[n].abs().max() == 0, n
            continue
        used += 1
        e = grads[n].reshape(g.shape)
        err = (e - g).abs().max() / g.abs().max().clamp_min(1e-30)
        assert err < 1e-4, "%s rel err %g" % (n, err)
    assert used > 50


def test_plan_structure():
    p = plan_mod.Plan(68, 8, 1, 8)
    assert len(p.ops) == 263                      # 264 conv calls per forward minus conv0 (SURVEY.md section 3.1)
    assert abs(p.conv_flops_per_image() / 1e9 - 22.116) < 1e-3     # BASELINE.md section 2
    assert plan_mod.Plan(68, 2, 1, 2).conv_flops_per_image() / 1e9 == pytest.approx(5.623, abs=1e-3)
    with pytest.raises(SystemExit):
        plan_mod.Plan(16, 2, 2, 2)                # order >= layer_num (models/cu_net.py:285-287)
    with pytest.raises(AssertionError):
        plan_mod.Plan(16, 2, 1, 3)                # loss_num > layer_num (models/cu_net.py:274)
    # every tensor's gradient accumulator has exactly one first writer and one last writer
    sched = p.backward_schedule()
    first, last = {}, {}
    for op, flags in sched:
        for (t, _), (acc, lst) in zip(op.srcs, flags):
            first[t.name] = first.get(t.name, 0) + (0 if acc else 1)
            last[t.name] = last.get(t.name, 0) + (1 if lst else 0)
    assert set(first.values()) == {1} and set(last.values()) == {1}
