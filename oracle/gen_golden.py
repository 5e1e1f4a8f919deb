"""Generate tests/golden/*.pt by executing the REAL reference (build container only).

    python -m oracle.gen_golden

TEST INFRASTRUCTURE -- see oracle/__init__.py.  The fixtures pin ``oracle/cunet_oracle.py`` and
``oracle/quantize_oracle.py`` to the reference's own behaviour (the reference ships no golden
vectors, SURVEY.md §4 / §8(c)).
"""
import os
import sys
import warnings

import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_loader, cunet_oracle, synthetic  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def run_reference(net, img, hm, train=True):
    net.train(train)
    net.zero_grad()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if train:
            outs = net(img)
            loss = cunet_oracle.multi_loss_mse(outs, hm)
            loss.backward()
        else:
            with torch.no_grad():
                outs = net(img)
                loss = cunet_oracle.multi_loss_mse(outs, hm)
    return outs, loss


def tiny_case(name, layer_num, order, loss_num, class_num, neck, growth, c0, seed):
    """Small-channel configuration: full tensors are stored."""
    torch.manual_seed(seed)
    net = ref_loader.create_reference_net(class_num, layer_num, order, loss_num,
                                          neck_size=neck, growth_rate=growth, init_chan_num=c0)
    state0 = {k: v.clone() for k, v in net.state_dict().items()}
    gen = torch.Generator().manual_seed(seed + 1)
    img = torch.rand(2, 3, 64, 64, generator=gen)
    hm = torch.rand(2, class_num, 16, 16, generator=gen)
    outs, loss = run_reference(net, img, hm, train=True)
    grads = {k: (p.grad.clone() if p.grad is not None else torch.zeros_like(p)) for k, p in net.named_parameters()}
    state1 = {k: v.clone() for k, v in net.state_dict().items()}
    outs_eval, loss_eval = run_reference(net, img, hm, train=False)
    torch.save({
        "config": dict(class_num=class_num, layer_num=layer_num, order=order, loss_num=loss_num,
                       neck_size=neck, growth_rate=growth, init_chan_num=c0),
        "state_before": state0, "img": img, "heatmap": hm,
        "outputs_train": [o.detach() for o in outs], "loss_train": loss.detach(),
        "grads": grads, "state_after_train": state1,
        "outputs_eval": [o.detach() for o in outs_eval], "loss_eval": loss_eval.detach(),
    }, os.path.join(OUT, name))


def real_case(name, layer_num, order, loss_num, class_num, n, seed):
    """Real channel configuration (4/32/128): digests only (weights are re-derivable from
    cunet_oracle.init_state(seed), inputs from synthetic.make_inputs(seed)).  Computed in float64: in float32 the
    small BatchNorm-weight gradients (sums that mostly cancel) move by up to ~2 % with the summation order of the
    host CPU, so a float32 digest only matches on a machine that sums like the one that recorded it."""
    state = cunet_oracle.init_state(class_num, layer_num, order, seed=seed)
    net = ref_loader.create_reference_net(class_num, layer_num, order, loss_num).double()
    missing = net.load_state_dict(state, strict=True)
    img, hm = (t.double() for t in synthetic.make_inputs(n, class_num, seed=seed))
    outs, loss = run_reference(net, img, hm, train=True)
    sd = net.state_dict()
    digest = {
        "config": dict(class_num=class_num, layer_num=layer_num, order=order, loss_num=loss_num,
                       n=n, seed=seed),
        "state_keys": list(sd.keys()),
        "state_shapes": [tuple(v.shape) for v in sd.values()],
        "loss_train": loss.detach(),
        "out_samples": [o.detach()[:, ::7, ::5, ::3].clone() for o in outs],
        "out_absmax": [o.detach().abs().max() for o in outs],
        "grad_norms": {k: p.grad.norm().clone() for k, p in net.named_parameters() if p.grad is not None},
        "grad_samples": {k: p.grad.flatten()[::97].clone() for k, p in net.named_parameters() if p.grad is not None},
        "running_mean_samples": {k: v.flatten()[::13].clone() for k, v in sd.items()
                                 if k.endswith("running_mean")},
        "running_var_samples": {k: v.flatten()[::13].clone() for k, v in sd.items()
                                if k.endswith("running_var")},
        "num_batches_tracked": {k: int(v) for k, v in sd.items() if k.endswith("num_batches_tracked")},
    }
    outs_eval, loss_eval = run_reference(net, img, hm, train=False)
    digest["loss_eval"] = loss_eval.detach()
    digest["out_eval_samples"] = [o.detach()[:, ::7, ::5, ::3].clone() for o in outs_eval]
    torch.save(digest, os.path.join(OUT, name))


def quant_case(name, bits_w, seed):
    """Run the real utils/quantize.py QuanOp on a small stack of Conv2d modules."""
    q = ref_loader.load_reference_quantize(bits_w)
    gen = torch.Generator().manual_seed(seed)
    shapes = [(8, 3, 3, 3), (32, 128, 3, 3), (16, 40, 1, 1), (32, 128, 3, 3), (5, 16, 1, 1), (4, 4, 1, 1)]
    convs = []
    for co, ci, k, _ in shapes:
        m = nn.Conv2d(ci, co, k, bias=False)
        m.weight.data = (torch.rand(co, ci, k, k, generator=gen) * 2 - 1) * 1.5
        convs.append(m)
    model = nn.Sequential(*convs)
    w0 = [m.weight.data.clone() for m in convs]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        op = q.QuanOp(model)
        op.quantization()
        wq = [m.weight.data.clone() for m in convs]
        grads = [torch.randn(m.weight.shape, generator=gen) * 0.01 for m in convs]
        for m, g in zip(convs, grads):
            m.weight.grad = g.clone()
        op.restore()
        wr = [m.weight.data.clone() for m in convs]
        op.updateQuanGradWeight()
        gq = [m.weight.grad.clone() for m in convs]
    torch.save({"bits_w": bits_w, "bits_g": 8, "w0": w0, "wq": wq, "wr": wr, "g0": grads, "gq": gq,
                "num_targets": op.num_of_params}, os.path.join(OUT, name))


def binop_case(name, seed):
    """Run the REAL BinOp (models/cu_net_prev_version.py:17-92, loaded by ref_loader.load_reference_binop) on a stack
    of Conv2d modules shaped like its target set in the prev-version model: conv0, dense-layer 3x3s, heads."""
    BinOp = ref_loader.load_reference_binop()
    gen = torch.Generator().manual_seed(seed)
    shapes = [(8, 3, 7, 7), (32, 128, 3, 3), (6, 128, 3, 3), (16, 128, 1, 1), (68, 128, 1, 1), (16, 128, 1, 1)]
    convs = []
    for co, ci, k, _ in shapes:
        m = nn.Conv2d(ci, co, k, bias=False)
        m.weight.data = (torch.rand(co, ci, k, k, generator=gen) * 2 - 1) * 1.5     # some |w| > 1: the clamp bites
        convs.append(m)
    model = nn.Sequential(*convs)
    w0 = [m.weight.data.clone() for m in convs]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        op = BinOp(model)
        op.binarization()
        wb = [m.weight.data.clone() for m in convs]
        grads = [torch.randn(m.weight.shape, generator=gen) * 0.01 for m in convs]
        for m, g in zip(convs, grads):
            m.weight.grad = g.clone()
        op.restore()
        wr = [m.weight.data.clone() for m in convs]
        op.updateBinaryGradWeight()
        gb = [m.weight.grad.clone() for m in convs]
    torch.save({"w0": w0, "wb": wb, "wr": wr, "g0": grads, "gb": gb, "num_targets": op.num_of_params},
               os.path.join(OUT, name))


def binop_targets_case(name):
    """Which tensors the reference's quantizers touch in the prev-version model (cu-net-prev-version-bin.py:50,65;
    cu-net-prev-version-wig.py:50,65): nn.Conv2d modules in modules() order with index 1 .. count-2.  The prev-version
    module cannot be constructed here (removed torch APIs), but its nn.Conv2d set is decided by three constructor
    sites only -- conv0 (cu_net_prev_version.py:451), one 3x3 ``conv.2`` per _DenseLayer (:170; the bottleneck 1x1 and
    every adapter are _EfficientDensenetBottleneck modules holding bare Parameters, :118-157, :166, :217-231, :294),
    one 1x1 ``conv`` per head (:348, ``layer_num`` heads :463-466) -- and by the registration order features, hg
    (down_blocks, up_blocks, neck_block :394-399), linears, intermedia (:450-470).  This builds a skeleton with exactly
    those Conv2d leaves in that order and lets the REAL BinOp constructor select from it."""
    BinOp = ref_loader.load_reference_binop()
    out = {}
    for L, class_num in ((2, 16), (8, 16), (8, 68)):
        root = nn.Module()
        root.features = nn.Sequential(nn.Conv2d(3, 128, 7, 2, 3, bias=False))
        hg = nn.Module()

        def block():
            b = nn.Module()
            b.layers = nn.ModuleList([nn.Sequential(nn.Conv2d(128, 32, 3, 1, 1, bias=False)) for _ in range(L)])
            return b
        hg.down_blocks = nn.ModuleList([block() for _ in range(4)])
        hg.up_blocks = nn.ModuleList([block() for _ in range(4)])
        hg.neck_block = block()
        root.hg = hg
        root.linears = nn.ModuleList([nn.Sequential(nn.Conv2d(128, class_num, 1, bias=False)) for _ in range(L)])
        names = {id(m.weight): n for n, m in root.named_modules() if isinstance(m, nn.Conv2d)}
        op = BinOp(root)
        out["L%d_C%d" % (L, class_num)] = dict(
            num_targets=op.num_of_params,
            shapes=[tuple(w.shape) for w in op.target_modules],
            names=[names[id(w)] for w in op.target_modules])
    torch.save(out, os.path.join(OUT, name))


def quaninput_case(name, seed):
    """QuanInput (utils/quantize.py:47-63): its forward / backward bodies are executed as plain functions of the real
    module (the legacy non-static autograd.Function cannot be *applied* on modern torch, but its two methods are
    ordinary python) with a stand-in ``self`` that implements save_for_backward / saved_tensors."""
    out = {}
    for bits_i in (8, 4):
        q = ref_loader.load_reference_quantize(1, bits_i=bits_i)
        gen = torch.Generator().manual_seed(seed + bits_i)
        x = torch.randn(4, 16, 8, 8, generator=gen) * 0.8
        x.view(-1)[:6] = torch.tensor([1.0, -1.0, 0.9921875, 0.99609375, 0.00390625, -0.01171875])   # edges / ties
        gy = torch.randn(x.shape, generator=gen)

        class Ctx(object):
            def save_for_backward(self, *t):
                self.saved_tensors = t
        ctx = Ctx()
        y = q.QuanInput.forward(ctx, x.clone())
        gx = q.QuanInput.backward(ctx, gy.clone())
        out[bits_i] = dict(x=x, y=y, gy=gy, gx=gx)
    torch.save(out, os.path.join(OUT, name))


def pylib_inputs(seed=11):
    """Seeded inputs of the validation-path fixture (shared with tests/test_oracle_golden.py)."""
    n, c = 3, 16
    _, target = synthetic.make_inputs(n, c, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    output = target + 0.2 * torch.randn(target.shape, generator=g)
    output[0, 3] = -1.0                      # no positive maximum: masked prediction
    target[1, 4] = 0.0                       # missing ground-truth joint
    output[2, 5] = 0.0
    output[2, 5, 0, 7] = 1.0                 # peak on the border: no quarter-pixel refinement
    center = torch.rand(n, 2, generator=g) * 400 + 300
    scale = torch.rand(n, generator=g) * 2 + 0.8
    rot = torch.tensor([0.0, 25.0, -40.0])
    pts = torch.rand(n, c, 2, generator=g) * 70 - 3
    pts[0, 0] = torch.tensor([2.5, 30.2])    # window start in (-1, 0): int() truncates towards zero
    pts[0, 1] = torch.tensor([63.9, 0.4])
    pts[0, 2] = torch.tensor([10.0, 12.0])
    pts[0, 3] = torch.tensor([66.2, 20.0])   # window partly inside from the right
    pts[0, 4] = torch.tensor([80.0, 20.0])   # entirely outside
    grnd = torch.rand(n, c, 2, generator=g) * 900 + 50
    grnd[0, 3] = 0.0
    norm = torch.rand(n, generator=g) * 20 + 40
    return dict(output=output, target=target, center=center, scale=scale, rot=rot, pts=pts, grnd_pts=grnd,
                normalizers=norm, idxs=[0, 1, 2, 3, 4, 5, 10, 11, 14, 15],
                flip_index=[[1, 4], [0, 5], [12, 13], [11, 14], [10, 15], [2, 3]])


def pylib_case(name):
    """Validation path + target heat maps: outputs of the REAL pylib/Evaluation.py, HumanAug.py, HumanPts.py."""
    import numpy as np
    mods = ref_loader.load_reference_pylib()
    ev, aug, hp = mods["Evaluation"], mods["HumanAug"], mods["HumanPts"]
    inp = pylib_inputs()
    out, tgt = inp["output"], inp["target"]
    res = [64, 64]
    # the big inputs are NOT stored: tests regenerate them with pylib_inputs() and check this fingerprint
    fx = dict(inputs_fingerprint=torch.stack([out.double().sum(), tgt.double().sum(), inp["pts"].double().sum()]),
              small_inputs={k: inp[k] for k in ("center", "scale", "rot", "grnd_pts", "normalizers", "idxs", "flip_index")})
    small = out[:2, :, 20:28, 20:28].contiguous()          # flip / shuffle are pure permutations: a crop pins them
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fx["get_preds"] = ev.get_preds(out.clone())
        fx["accuracy"] = ev.accuracy(out.clone(), tgt.clone(), inp["idxs"])
        fx["final_preds"] = ev.final_preds(out.clone(), inp["center"], inp["scale"], res, inp["rot"])
        fx["accuracy_origin_res"] = ev.accuracy_origin_res(out.clone(), inp["center"], inp["scale"], res,
                                                           inp["grnd_pts"], inp["normalizers"], inp["rot"])
        fx["calc_dists"] = ev.calc_dists(fx["final_preds"], inp["grnd_pts"], inp["normalizers"], use_zero=True)
        fx["flip_channels"] = aug.flip_channels(small.clone())
        fx["shuffle"] = aug.shuffle_channels_for_horizontal_flipping(small.clone(), np.array(inp["flip_index"]))
        h, v = hp.pts2heatmap(inp["pts"][0].numpy().astype(np.float64), (64, 64), 1)     # sample 0 holds the edge cases
        fx["pts2heatmap"], fx["valid_pts"] = torch.from_numpy(h).float(), torch.from_numpy(v)
        # hp.heatmap2pts is not executed: it relies on torch-0.1.12's keepdim=True result of torch.max (HumanPts.py:94,104)
    torch.save(fx, os.path.join(OUT, name))


def history_updates():
    """The TrainHistory.update() arguments of the checkpoint fixture (shared with tests/test_checkpoint_cpu.py)."""
    from collections import OrderedDict
    return [(OrderedDict([("epoch", e)]), OrderedDict([("lr", lr)]),
             OrderedDict([("train_loss", 1.0 / (e + 1)), ("val_loss", 2.0 / (e + 1))]), OrderedDict([("val_pckh", pck)]))
            for e, (pck, lr) in enumerate([(0.1, 1e-3), (0.3, 1e-3), (0.2, 5e-4)])]


def checkpoint_case(name):
    """Checkpoint bookkeeping of the REAL reference: TrainHistory (utils/util.py:8-46) over history_updates(), the keys
    its load_state_dict reads, adjust_lr (utils/util.py:106-119) over 200 epochs, and the parameter trees of its
    create_cu_net (state_dict names / shapes / dtypes; nn.Conv2d modules in modules() order)."""
    import contextlib
    import io
    import types
    util = ref_loader.load_reference_util()
    hist = util["TrainHistory"]()
    steps = []
    for args in history_updates():
        hist.update(*args)
        steps.append((hist.is_best, hist.best_pckh))

    class Recorder(dict):
        def __getitem__(self, k):
            self.read.append(k)
            return dict.__getitem__(self, k)
    rec = Recorder(hist.state_dict())
    rec.read = []
    util["TrainHistory"]().load_state_dict(rec)
    opt = types.SimpleNamespace(lr=2.5e-4)
    optimizer = types.SimpleNamespace(param_groups=[{"lr": 2.5e-4}])
    lrs = []
    with contextlib.redirect_stdout(io.StringIO()):
        for e in range(200):
            util["adjust_lr"](opt, optimizer, e)
            lrs.append(opt.lr)
    net = ref_loader.create_reference_net(5, 3, 1, 2)
    tree = [(k, tuple(v.shape), v.dtype) for k, v in net.state_dict().items()]
    net = ref_loader.create_reference_net(5, 3, 2, 3)
    convs = [(n, tuple(m.weight.shape)) for n, m in net.named_modules() if isinstance(m, nn.Conv2d)]
    torch.save({"history_steps": steps, "history_state": hist.state_dict(), "history_load_keys": rec.read,
                "adjust_lr": lrs, "state_tree_C5_L3_K1_loss2": tree, "convs_C5_L3_K2_loss3": convs},
               os.path.join(OUT, name))


def cross_check_inputs():
    """Seeded inputs of cross_check.pt (tests regenerate them and check the fixture's fingerprint):
    CU-Net weights (cunet_oracle.init_state) and a batch for class_num 4, layer_num 3, order 1, neck 2, growth 8,
    16 initial channels; weights and gradients of a four-conv stack for BinOp."""
    state = cunet_oracle.init_state(4, 3, 1, seed=5, neck_size=2, growth_rate=8, init_chan_num=16)
    gen = torch.Generator().manual_seed(6)
    img, hm = torch.rand(2, 3, 64, 64, generator=gen), torch.rand(2, 4, 16, 16, generator=gen)
    gen = torch.Generator().manual_seed(77)
    shapes = [(4, 3, 3, 3), (32, 128, 3, 3), (16, 128, 1, 1), (4, 4, 1, 1)]
    w0 = [(torch.rand(s, generator=gen) * 2 - 1) * 1.2 for s in shapes]
    g0 = [torch.randn(s, generator=gen) for s in shapes]
    return dict(state=state, img=img, heatmap=hm, binop_w0=w0, binop_g0=g0)


def input_fingerprint(inp):
    return torch.stack([t.double().sum() for t in [inp["img"], inp["heatmap"]] + list(inp["state"].values())
                        + inp["binop_w0"] + inp["binop_g0"]])


CROSS_STRIDE = 8      # every 8th element of each gradient / binarised weight is stored (the file stays small)


def cross_check_case(name):
    """Outputs of the REAL reference on inputs the other fixtures do not cover: loss and gradients of a CU-Net with
    three losses (models/cu_net.py), BinOp (models/cu_net_prev_version.py:17-92) on a four-conv stack, and the
    validation path (pylib/Evaluation.py, HumanAug.GetTransform) on pylib_inputs(seed=23)."""
    import numpy as np
    inp = cross_check_inputs()
    net = ref_loader.create_reference_net(4, 3, 1, 3, neck_size=2, growth_rate=8, init_chan_num=16).double()
    net.load_state_dict(inp["state"], strict=True)
    _, loss = run_reference(net, inp["img"].double(), inp["heatmap"].double(), train=True)     # float64: see real_case
    names = [k for k, _ in net.named_parameters()]
    grads = torch.cat([p.grad.flatten()[::CROSS_STRIDE] for _, p in net.named_parameters()])
    BinOp = ref_loader.load_reference_binop()
    convs = [nn.Conv2d(w.shape[1], w.shape[0], w.shape[2], bias=False) for w in inp["binop_w0"]]
    for m, w in zip(convs, inp["binop_w0"]):
        m.weight.data = w.clone()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        op = BinOp(nn.Sequential(*convs))
        op.binarization()
        wb = [m.weight.data.flatten()[::CROSS_STRIDE].clone() for m in convs]
        for m, g in zip(convs, inp["binop_g0"]):
            m.weight.grad = g.clone()
        op.restore()
        op.updateBinaryGradWeight()
        gb = [m.weight.grad.flatten()[::CROSS_STRIDE].clone() for m in convs]
    mods = ref_loader.load_reference_pylib()
    pin = pylib_inputs(seed=23)
    out, tgt, res = pin["output"], pin["target"], [64, 64]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pylib = dict(get_preds=mods["Evaluation"].get_preds(out.clone()),
                     accuracy=mods["Evaluation"].accuracy(out.clone(), tgt.clone(), pin["idxs"]),
                     final_preds=mods["Evaluation"].final_preds(out.clone(), pin["center"], pin["scale"], res, pin["rot"]),
                     transform=torch.from_numpy(np.asarray(
                         mods["HumanAug"].GetTransform(np.array([320.0, 410.0]), 1.7, 30.0, 64, 200), dtype=np.float64)))
    torch.save({"inputs_fingerprint": input_fingerprint(inp), "stride": CROSS_STRIDE,
                "cunet_loss": loss.detach(), "cunet_param_names": names, "cunet_grads": grads, "binop_num_targets": op.num_of_params,
                "binop_wb": wb, "binop_gb": gb,
                "pylib_fingerprint": torch.stack([out.double().sum(), tgt.double().sum()]), "pylib": pylib},
               os.path.join(OUT, name))


def main():
    os.makedirs(OUT, exist_ok=True)
    checkpoint_case("checkpoint_ref.pt")
    cross_check_case("cross_check.pt")
    pylib_case("pylib_eval.pt")
    tiny_case("tiny_L3_K2.pt", 3, 2, 2, 5, 2, 8, 16, seed=11)
    tiny_case("tiny_L2_K1.pt", 2, 1, 2, 3, 4, 8, 16, seed=12)
    tiny_case("tiny_L3_K0.pt", 3, 0, 3, 4, 2, 8, 16, seed=13)
    real_case("real_L2_K1_C68_n1.pt", 2, 1, 2, 68, 1, seed=0)
    for bw in (1, 2, 8):
        quant_case("quanop_bits%d.pt" % bw, bw, seed=20 + bw)
    binop_case("binop.pt", seed=31)
    binop_targets_case("binop_targets.pt")
    quaninput_case("quaninput.pt", seed=41)
    print("golden fixtures written to", OUT)


if __name__ == "__main__":
    main()
