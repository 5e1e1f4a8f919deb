"""Pins the CPU oracle (oracle/*.py) to the reference's own behaviour.

Fixtures in tests/golden/ were produced by the REAL reference (oracle/gen_golden.py); the tests need only them.
The ``*_live_against_reference`` tests keep their names from when they executed the reference side by side: they now
compare against its outputs recorded in tests/golden/cross_check.pt, and nothing here runs the reference.
"""
import os

import pytest
import torch

from oracle import cunet_oracle, quantize_oracle, evaluation_oracle, synthetic

TINY = ["tiny_L3_K2.pt", "tiny_L2_K1.pt", "tiny_L3_K0.pt"]


def _close(a, b, tol=2e-5):
    a, b = a.double(), b.double()
    scale = max(b.abs().max().item(), 1e-12)
    return (a - b).abs().max().item() / scale <= tol


@pytest.mark.parametrize("name", TINY)
def test_oracle_matches_reference_fixture(golden_dir, name):
    fx = torch.load(os.path.join(golden_dir, name), weights_only=False)
    cfg = fx["config"]
    net = cunet_oracle.OracleCUNet(fx["state_before"], cfg["class_num"], cfg["layer_num"],
                                   cfg["order"], cfg["loss_num"], neck_size=cfg["neck_size"],
                                   growth_rate=cfg["growth_rate"], init_chan_num=cfg["init_chan_num"])
    spec_names = [n for n, _, _ in cunet_oracle.state_spec(
        cfg["class_num"], cfg["layer_num"], cfg["order"], cfg["neck_size"], cfg["growth_rate"],
        cfg["init_chan_num"])]
    assert spec_names == list(fx["state_before"].keys())        # names + registration order
    for (n, shape, _), v in zip(cunet_oracle.state_spec(
            cfg["class_num"], cfg["layer_num"], cfg["order"], cfg["neck_size"],
            cfg["growth_rate"], cfg["init_chan_num"]), fx["state_before"].values()):
        assert tuple(v.shape) == tuple(shape), n
    net.train()
    outs = net(fx["img"])
    loss = cunet_oracle.multi_loss_mse(outs, fx["heatmap"])
    loss.backward()
    assert len(outs) == len(fx["outputs_train"])
    for o, r in zip(outs, fx["outputs_train"]):
        assert _close(o.detach(), r)
    assert _close(loss.detach(), fx["loss_train"])
    for n in net.param_names:
        g = net.state[n].grad
        g = torch.zeros_like(net.state[n]) if g is None else g
        assert _close(g, fx["grads"][n], 2e-4), n
    # BN running statistics incl. the double update of checkpointed BNs (SURVEY §8 A9)
    for k, v in fx["state_after_train"].items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert _close(net.state[k], v, 1e-5), k
        if k.endswith("num_batches_tracked"):
            assert int(net.state[k]) == int(v), k
    net.eval()
    with torch.no_grad():
        outs = net(fx["img"])
    for o, r in zip(outs, fx["outputs_eval"]):
        assert _close(o, r)


def test_oracle_real_config_digest(golden_dir):
    fx = torch.load(os.path.join(golden_dir, "real_L2_K1_C68_n1.pt"), weights_only=False)
    cfg = fx["config"]
    state = cunet_oracle.init_state(cfg["class_num"], cfg["layer_num"], cfg["order"], seed=cfg["seed"])
    assert list(state.keys()) == fx["state_keys"]
    assert [tuple(v.shape) for v in state.values()] == fx["state_shapes"]
    assert len(state) == 396                                      # SURVEY.md §8(b)
    # float64 on both sides (oracle/gen_golden.real_case): the comparison does not depend on the CPU's summation order
    net = cunet_oracle.OracleCUNet({k: v.double() if v.is_floating_point() else v for k, v in state.items()},
                                   cfg["class_num"], cfg["layer_num"], cfg["order"], cfg["loss_num"])
    for n in net.param_names:
        net.state[n] = net.state[n].detach().double().requires_grad_(True)
    img, hm = (t.double() for t in synthetic.make_inputs(cfg["n"], cfg["class_num"], seed=cfg["seed"]))
    outs = net(img)
    loss = cunet_oracle.multi_loss_mse(outs, hm)
    loss.backward()
    assert _close(loss.detach(), fx["loss_train"], 1e-5)
    for o, r in zip(outs, fx["out_samples"]):
        assert _close(o.detach()[:, ::7, ::5, ::3], r, 1e-4)
    for k, r in fx["grad_samples"].items():
        assert _close(net.state[k].grad.flatten()[::97], r, 1e-3), k
    for k, r in fx["running_var_samples"].items():
        assert _close(net.state[k].flatten()[::13], r, 1e-5), k
    for k, r in fx["num_batches_tracked"].items():
        assert int(net.state[k]) == r, k


def _cross_check_fixture(golden_dir):
    from oracle import gen_golden
    fx = torch.load(os.path.join(golden_dir, "cross_check.pt"), weights_only=False)
    inp = gen_golden.cross_check_inputs()
    assert torch.allclose(gen_golden.input_fingerprint(inp), fx["inputs_fingerprint"], rtol=0, atol=1e-9), \
        "seeded inputs drifted from the fixture's"
    return fx, inp


def test_oracle_against_live_reference(golden_dir):
    """Loss and gradients of the oracle against the reference's (tests/golden/cross_check.pt, float64) on a
    configuration none of the other fixtures has: order 1, three losses, neck 2, growth 8, 16 initial channels."""
    fx, inp = _cross_check_fixture(golden_dir)
    net = cunet_oracle.OracleCUNet({k: v.double() if v.is_floating_point() else v for k, v in inp["state"].items()},
                                   4, 3, 1, 3, neck_size=2, growth_rate=8, init_chan_num=16)
    for n in net.param_names:                      # float64 on both sides, like test_oracle_real_config_digest
        net.state[n] = net.state[n].detach().double().requires_grad_(True)
    ol = cunet_oracle.multi_loss_mse(net(inp["img"].double()), inp["heatmap"].double())
    ol.backward()
    assert _close(ol.detach(), fx["cunet_loss"])
    assert net.param_names == fx["cunet_param_names"]
    at = 0
    for n in net.param_names:
        g = net.state[n].grad.flatten()[::fx["stride"]]
        assert _close(g, fx["cunet_grads"][at:at + g.numel()], 2e-4), n
        at += g.numel()
    assert at == fx["cunet_grads"].numel()


@pytest.mark.parametrize("bits_w", [1, 2, 8])
def test_quanop_oracle_matches_reference_fixture(golden_dir, bits_w):
    fx = torch.load(os.path.join(golden_dir, "quanop_bits%d.pt" % bits_w), weights_only=False)
    idx = quantize_oracle.target_indices(len(fx["w0"]))
    assert len(idx) == fx["num_targets"]
    tw = [fx["w0"][i] for i in idx]
    wq, saved = quantize_oracle.quanop_quantization(tw, bits_w, fx["bits_g"])
    for j, i in enumerate(idx):
        assert torch.equal(wq[j], fx["wq"][i]), (bits_w, i)
        assert torch.equal(saved[j], fx["wr"][i]), (bits_w, i)
    for i in range(len(fx["w0"])):                 # first / last conv untouched
        if i not in idx:
            assert torch.equal(fx["wq"][i], fx["w0"][i])
    gq = quantize_oracle.quanop_update_grad(saved, [fx["g0"][i] for i in idx], bits_w, fx["bits_g"])
    for j, i in enumerate(idx):
        assert torch.equal(gq[j], fx["gq"][i]), (bits_w, i)
    # value sets (SURVEY.md §8 A12)
    if bits_w in (1, 2):
        for w in wq:
            assert set(w.unique().tolist()) <= {-1.0, 0.0, 1.0}
    for g in gq:
        assert torch.equal(g * 128, torch.round(g * 128)) and g.abs().max() <= 0.9921875


def test_binop_oracle_matches_reference_fixture(golden_dir):
    """oracle/quantize_oracle.binop_* against the outputs of the REAL BinOp (models/cu_net_prev_version.py:17-92,
    executed by oracle/gen_golden.binop_case through ref_loader.load_reference_binop)."""
    fx = torch.load(os.path.join(golden_dir, "binop.pt"), weights_only=False)
    idx = quantize_oracle.target_indices(len(fx["w0"]))
    assert len(idx) == fx["num_targets"]
    wb, saved = quantize_oracle.binop_binarization([fx["w0"][i] for i in idx])
    for j, i in enumerate(idx):
        assert _close(wb[j], fx["wb"][i], 1e-6), i
        assert torch.equal(wb[j].sign(), fx["wb"][i].sign()), i
        assert _close(saved[j], fx["wr"][i], 1e-7), i
    for i in range(len(fx["w0"])):                 # first / last conv untouched
        if i not in idx:
            assert torch.equal(fx["wb"][i], fx["w0"][i]) and torch.equal(fx["gb"][i], fx["g0"][i])
    gb = quantize_oracle.binop_update_grad([fx["wr"][i] for i in idx], [fx["g0"][i] for i in idx])
    for j, i in enumerate(idx):
        assert _close(gb[j], fx["gb"][i], 1e-4), i


def test_binop_oracle_live_against_reference(golden_dir):
    """oracle/quantize_oracle.binop_* against the REAL BinOp's binarised weights and fixed gradients on a second conv
    stack (tests/golden/cross_check.pt)."""
    fx, inp = _cross_check_fixture(golden_dir)
    w0, g0, k = inp["binop_w0"], inp["binop_g0"], fx["stride"]
    idx = quantize_oracle.target_indices(len(w0))
    assert idx == [1, 2] and len(idx) == fx["binop_num_targets"]
    wb, saved = quantize_oracle.binop_binarization([w0[i] for i in idx])
    for a, i in zip(wb, idx):
        assert _close(a.flatten()[::k], fx["binop_wb"][i], 1e-6), i
    for a, i in zip(quantize_oracle.binop_update_grad(saved, [g0[i] for i in idx]), idx):
        assert _close(a.flatten()[::k], fx["binop_gb"][i], 1e-4), i
    for i in (0, 3):                               # first / last conv untouched
        assert torch.equal(w0[i].flatten()[::k], fx["binop_wb"][i]) and torch.equal(g0[i].flatten()[::k], fx["binop_gb"][i])


@pytest.mark.parametrize("cfg", [(2, 16), (8, 16), (8, 68)])
def test_quantizer_target_set_is_the_prev_version_set(golden_dir, cfg):
    """BASELINE.json configs[3]: the tensors BinOp / QuanOp select on the drop-in module are the ones the REAL BinOp
    constructor selects on the prev-version model's nn.Conv2d skeleton (tests/golden/binop_targets.pt): for L=8 the
    72 dense-layer 3x3 convs + 7 of the 8 heads, not the 262 convs of the drop-in tree."""
    from cunet_b200.models.cu_net import create_cu_net
    from cunet_b200.utils.quantize import target_names
    L, C = cfg
    fx = torch.load(os.path.join(golden_dir, "binop_targets.pt"), weights_only=False)["L%d_C%d" % (L, C)]
    net = create_cu_net(4, 32, 128, C, L, 1, L)
    names = target_names(net)                                  # default for a CU-Net drop-in: prev_version
    mods = dict(net.named_modules())
    assert len(names) == fx["num_targets"] == 9 * L + L - 1
    assert [tuple(mods[n].weight.shape) for n in names] == fx["shapes"]
    skeleton = [n[:-len("conv2")] + "0" if n.endswith("conv2") else n[:-len("conv")] + "0" for n in names]
    assert skeleton == fx["names"]
    assert len(target_names(net, "all_conv2d")) == 33 * L - 2


def test_quaninput_oracle_matches_reference_fixture(golden_dir):
    """quantize_oracle.quan_input_* against the REAL QuanInput.forward / .backward bodies (utils/quantize.py:47-63)."""
    fx = torch.load(os.path.join(golden_dir, "quaninput.pt"), weights_only=False)
    for bits_i, d in fx.items():
        assert torch.equal(quantize_oracle.quan_input_forward(d["x"], bits_i), d["y"])
        assert torch.equal(quantize_oracle.quan_input_backward(d["x"], d["gy"]), d["gx"])
        sc = 2.0 ** (bits_i - 1)
        assert torch.equal(d["y"] * sc, torch.round(d["y"] * sc)) and d["y"].abs().max() <= 1 - 1 / sc


def test_binop_properties():
    gen = torch.Generator().manual_seed(3)
    w = [(torch.rand(32, 128, 3, 3, generator=gen) * 2 - 1) * 1.3]
    wb, saved = quantize_oracle.binop_binarization(w)
    s = saved[0]
    assert s.abs().max() <= 1.0
    alpha = s.abs().mean(dim=(1, 2, 3), keepdim=True)
    assert torch.allclose(wb[0], s.sign() * alpha)
    g = [torch.randn(32, 128, 3, 3, generator=gen)]
    gu = quantize_oracle.binop_update_grad(saved, g)[0]
    n = 128 * 9
    expect = (alpha * (s.abs() <= 1).float() * g[0]
              + s.sign() * (s.sign() * g[0]).sum(dim=(1, 2, 3), keepdim=True) / n) * (1 - 1 / 128.) * n
    assert torch.allclose(gu, expect, rtol=1e-5, atol=1e-6)


def test_get_preds_semantics():
    s = torch.zeros(1, 3, 64, 64)
    s[0, 0, 10, 20] = 2.0
    s[0, 0, 30, 40] = 2.0        # tie -> first maximum
    s[0, 1] = -1.0               # max <= 0 -> masked
    s[0, 2, 63, 63] = 0.5
    p = evaluation_oracle.get_preds(s)
    assert p[0, 0].tolist() == [21.0, 11.0]
    assert p[0, 1].tolist() == [0.0, 0.0]
    assert p[0, 2].tolist() == [64.0, 64.0]
    img, hm = synthetic.make_inputs(2, 5, seed=1)
    p = evaluation_oracle.get_preds(hm)
    assert (p >= 5).all() and (p <= 60).all()


def test_product_synthetic_matches_oracle_copy():
    """cu-net.py / bench.py generate their batches with cunet_b200.utils.synthetic; the oracle keeps its own copy."""
    from cunet_b200.utils import synthetic as prod
    for seed in (0, 7):
        a, b = prod.make_inputs(2, 5, seed=seed), synthetic.make_inputs(2, 5, seed=seed)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ---- validation path + target heat maps: oracle/evaluation_oracle.py against the REAL pylib functions -----------------
def _pylib_fixture(golden_dir):
    from oracle import gen_golden
    fx = torch.load(os.path.join(golden_dir, "pylib_eval.pt"), weights_only=False)
    inp = gen_golden.pylib_inputs()
    fp = torch.stack([inp["output"].double().sum(), inp["target"].double().sum(), inp["pts"].double().sum()])
    assert torch.allclose(fp, fx["inputs_fingerprint"], rtol=0, atol=1e-9), "seeded inputs drifted from the fixture's"
    return fx, inp


def test_evaluation_oracle_matches_reference_fixture(golden_dir):
    """get_preds / accuracy / final_preds / accuracy_origin_res / calc_dists of pylib/Evaluation.py, flip helpers of
    pylib/HumanAug.py and pts2heatmap of pylib/HumanPts.py: outputs recorded from the real reference functions."""
    import numpy as np
    fx, inp = _pylib_fixture(golden_dir)
    out, tgt, res = inp["output"], inp["target"], [64, 64]
    assert torch.equal(evaluation_oracle.get_preds(out), fx["get_preds"])
    assert torch.allclose(evaluation_oracle.accuracy(out, tgt, inp["idxs"]), fx["accuracy"], atol=1e-7)
    fp = evaluation_oracle.final_preds(out.clone(), inp["center"], inp["scale"], res, inp["rot"])
    assert torch.equal(fp, fx["final_preds"])
    assert torch.allclose(evaluation_oracle.calc_dists(fp, inp["grnd_pts"], inp["normalizers"], use_zero=True),
                          fx["calc_dists"], atol=1e-6)
    assert torch.allclose(evaluation_oracle.accuracy_origin_res(out.clone(), inp["center"], inp["scale"], res,
                                                                inp["grnd_pts"], inp["normalizers"], inp["rot"]),
                          fx["accuracy_origin_res"], atol=1e-7)
    small = out[:2, :, 20:28, 20:28].contiguous()
    assert torch.equal(evaluation_oracle.flip_channels(small.clone()), fx["flip_channels"])
    assert torch.equal(evaluation_oracle.shuffle_channels_for_horizontal_flipping(small.clone(), inp["flip_index"]),
                       fx["shuffle"])
    h, v = evaluation_oracle.pts2heatmap(inp["pts"][0].numpy().astype(np.float64), (64, 64), 1)
    assert np.abs(h - fx["pts2heatmap"].numpy()).max() < 1e-6 and np.abs(v - fx["valid_pts"].numpy()).max() == 0


def test_product_validation_dropins_match_reference_fixture(golden_dir):
    """The vectorised drop-ins of cunet_b200.pylib (device-agnostic arithmetic) against the same recorded outputs."""
    from cunet_b200.pylib import Evaluation, HumanAug, HumanPts
    fx, inp = _pylib_fixture(golden_dir)
    out, tgt, res = inp["output"], inp["target"], [64, 64]
    preds, gts = fx["get_preds"], evaluation_oracle.get_preds(tgt)
    assert torch.allclose(Evaluation.accuracy_from_preds(preds, gts, 64, inp["idxs"]), fx["accuracy"], atol=1e-6)
    got = Evaluation.final_preds_from_coords(out, preds, inp["center"], inp["scale"], res, inp["rot"])
    assert (got - fx["final_preds"]).abs().max() <= 1.0 and ((got - fx["final_preds"]).abs() > 0).float().mean() < 0.03
    assert torch.allclose(Evaluation.calc_dists(fx["final_preds"], inp["grnd_pts"], inp["normalizers"], use_zero=True),
                          fx["calc_dists"], atol=1e-5)
    small = out[:2, :, 20:28, 20:28].contiguous()
    assert torch.equal(HumanAug.flip_channels(small), fx["flip_channels"])
    assert torch.equal(HumanAug.shuffle_channels_for_horizontal_flipping(small, inp["flip_index"]), fx["shuffle"])
    hm, valid = HumanPts.pts2heatmap(inp["pts"][0], (64, 64), 1)
    assert (hm - fx["pts2heatmap"]).abs().max() < 1e-6 and (valid.double() - fx["valid_pts"]).abs().max() < 1e-6


def test_evaluation_oracle_live_against_reference(golden_dir):
    """The oracle's validation path against the real pylib functions' outputs on a second seed
    (tests/golden/cross_check.pt; pylib_eval.pt holds the first)."""
    import numpy as np
    from oracle import gen_golden
    fx = torch.load(os.path.join(golden_dir, "cross_check.pt"), weights_only=False)
    ref = fx["pylib"]
    inp = gen_golden.pylib_inputs(seed=23)
    out, tgt, res = inp["output"], inp["target"], [64, 64]
    fp = torch.stack([out.double().sum(), tgt.double().sum()])
    assert torch.allclose(fp, fx["pylib_fingerprint"], rtol=0, atol=1e-9), "seeded inputs drifted from the fixture's"
    assert torch.equal(evaluation_oracle.get_preds(out), ref["get_preds"])
    assert torch.allclose(evaluation_oracle.accuracy(out, tgt, inp["idxs"]), ref["accuracy"], atol=1e-7)
    assert torch.equal(evaluation_oracle.final_preds(out.clone(), inp["center"], inp["scale"], res, inp["rot"]),
                       ref["final_preds"])
    t = evaluation_oracle.get_transform(np.array([320.0, 410.0]), 1.7, 30.0, 64, 200)
    assert np.abs(t - ref["transform"].numpy()).max() < 1e-12
