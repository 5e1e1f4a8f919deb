"""Checkpoint compatibility with the reference (utils/checkpoint.py:40-67), host logic only (no GPU):
the parameter tree of cunet_b200's CUNetB200 carries the reference's names and NCHW shapes, so a state_dict written
by the reference's DataParallel-wrapped net loads by name, and files written here load in the reference."""
import os
from collections import OrderedDict

import pytest
import torch


def _History(lr=2.5e-4, epoch=3):
    """The product's TrainHistory (drop-in for utils/util.py:8-46) holding one epoch record."""
    from collections import OrderedDict
    from cunet_b200.utils.util import TrainHistory
    h = TrainHistory()
    h.update(OrderedDict([("epoch", epoch)]), OrderedDict([("lr", lr)]),
             OrderedDict([("train_loss", 0.5), ("val_loss", 0.6)]), OrderedDict([("val_pckh", 0.25)]))
    return h


def _reference(golden_dir):
    """What the reference's own code recorded (oracle/gen_golden.checkpoint_case): TrainHistory bookkeeping, the keys
    its load_state_dict reads, adjust_lr over 200 epochs, and the parameter trees of its create_cu_net."""
    return torch.load(os.path.join(golden_dir, "checkpoint_ref.pt"), weights_only=False)


def test_train_history_round_trips_with_the_reference_class(tmp_path, golden_dir):
    """A checkpoint's 'train_history' written here loads in the reference's TrainHistory.load_state_dict
    (utils/util.py:40-46: epoch, lr, loss, pckh, best_pckh, is_best) and vice versa, with identical bookkeeping."""
    from cunet_b200.utils.util import TrainHistory
    from oracle import gen_golden
    ref = _reference(golden_dir)
    ours = TrainHistory()
    for args, (is_best, best_pckh) in zip(gen_golden.history_updates(), ref["history_steps"]):
        ours.update(*args)
        assert ours.is_best == is_best and ours.best_pckh == best_pckh
    assert list(ours.state_dict().keys()) == list(ref["history_state"].keys())
    assert ours.state_dict() == ref["history_state"]
    path = str(tmp_path / "h.pt")
    torch.save({"train_history": ours.state_dict()}, path)
    back = torch.load(path, weights_only=False)["train_history"]
    assert {k: back[k] for k in ref["history_load_keys"]} == {k: ref["history_state"][k] for k in ref["history_load_keys"]}
    mine = TrainHistory()
    mine.load_state_dict(ref["history_state"])
    assert mine.state_dict() == ours.state_dict() and mine.last_epoch() == 2
    assert TrainHistory().last_epoch() == -1                                            # empty: no sentinel records


def _nets(golden_dir):
    """Ours and the reference's state_dict (zeros, in the reference's names / order / shapes / dtypes) for class_num 5,
    layer_num 3, order 1, loss_num 2."""
    from cunet_b200.models.cu_net import create_cu_net
    ours = create_cu_net(4, 32, 128, 5, 3, 1, 2)
    ref_sd = OrderedDict((k, torch.zeros(shape, dtype=dt)) for k, shape, dt in _reference(golden_dir)["state_tree_C5_L3_K1_loss2"])
    return ours, ref_sd


def test_reference_checkpoint_loads_by_name(tmp_path, golden_dir):
    from cunet_b200.utils.checkpoint import Checkpoint
    ours, ref_sd = _nets(golden_dir)
    assert list(ref_sd.keys()) == list(ours.state_dict().keys())          # names and registration order
    # what the reference writes: DataParallel-prefixed keys + RMSprop state (cu-net.py:59-61, utils/checkpoint.py:16-19)
    torch.manual_seed(1)
    for v in ref_sd.values():
        if v.dtype.is_floating_point:
            v.copy_(torch.randn_like(v))
    params = [torch.nn.Parameter(v) for k, v in ref_sd.items() if not k.endswith(("running_mean", "running_var",
                                                                                  "num_batches_tracked"))]
    opt = torch.optim.RMSprop(params, lr=1e-3, alpha=0.99, eps=1e-8)
    path = str(tmp_path / "lr-0.001-7")
    torch.save({"train_history": {"lr": [{"lr": 1e-3}], "epoch": [{"epoch": 7}]},
                "state_dict": {"module." + k: v for k, v in ref_sd.items()},
                "optimizer": opt.state_dict()}, path + ".pth.tar")
    ck = Checkpoint()
    ck.load_prefix = path
    hist = _History()
    assert ck.load_checkpoint(ours, None, hist)
    assert hist.epoch[-1]["epoch"] == 7
    for k, v in ours.state_dict().items():
        assert torch.equal(v, ref_sd[k]), k


def test_our_checkpoint_loads_in_the_reference(tmp_path, golden_dir):
    from cunet_b200.utils.checkpoint import Checkpoint
    ours, ref_sd = _nets(golden_dir)
    ck = Checkpoint()
    ck.save_prefix = str(tmp_path) + os.sep
    opt = torch.optim.RMSprop(ours.parameters(), lr=2.5e-4, alpha=0.99, eps=1e-8)
    path = ck.save_checkpoint(ours, opt, _History(2.5e-4, 3))
    assert path.endswith("lr-0.00025-3.pth.tar") and os.path.isfile(path[:-8] + "-model-best.pth.tar")
    saved = torch.load(path, weights_only=False)
    assert all(k.startswith("module.") for k in saved["state_dict"])
    # the reference's own loop (utils/checkpoint.py:53-61) on its DataParallel-named dict
    net_dict = {"module." + k: v for k, v in ref_sd.items()}
    for name, param in saved["state_dict"].items():
        assert name in net_dict, name
        assert param.shape == net_dict[name].shape and param.dtype == net_dict[name].dtype, name
        net_dict[name].copy_(param)
    for k, v in ours.state_dict().items():
        assert torch.equal(ref_sd[k], v), k


def test_old_checkpoints_without_num_batches_tracked(tmp_path):
    from cunet_b200.models.cu_net import create_cu_net
    from cunet_b200.utils.checkpoint import load_weights
    a = create_cu_net(4, 32, 128, 3, 2, 1, 2)
    b = create_cu_net(4, 32, 128, 3, 2, 1, 2)
    sd = {"module." + k: v for k, v in a.state_dict().items() if not k.endswith("num_batches_tracked")}
    sd["module.not_in_net.weight"] = torch.zeros(1)
    loaded, skipped, missing = load_weights(b, sd)
    assert skipped == ["not_in_net.weight"] and all(m.endswith("num_batches_tracked") for m in missing)
    for k, v in b.state_dict().items():
        if not k.endswith("num_batches_tracked"):
            assert torch.equal(v, a.state_dict()[k]), k
    with pytest.raises(ValueError):
        load_weights(b, {"features.conv0.weight": torch.zeros(2, 2)})


def test_entry_point_resume(tmp_path):
    """cu-net.py --resume_prefix: weights, lr and epoch come back from a checkpoint in the reference's format."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("cu_net_entry", os.path.join(root, "cu-net.py"))
    entry = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(entry)
    from cunet_b200.models.cu_net import create_cu_net
    from cunet_b200.utils.checkpoint import Checkpoint
    a = create_cu_net(4, 32, 128, 3, 2, 1, 2)
    hist = _History(5e-4, 11)
    os.makedirs(str(tmp_path / "run1"))
    ck = Checkpoint()
    ck.save_prefix = str(tmp_path / "run1") + os.sep
    opt_a = torch.optim.RMSprop(a.parameters(), lr=5e-4)
    path = ck.save_checkpoint(a, opt_a, hist)
    opt = entry.parse(["--exp_dir", str(tmp_path), "--exp_id", "run1", "--layer_num", "2", "--class_num", "3",
                       "--resume_prefix", os.path.basename(path)])
    b = create_cu_net(4, 32, 128, 3, 2, 1, 2)
    hist_b = entry.TrainHistory()
    state = entry.resume(b, opt, hist_b)
    assert opt.lr == 5e-4 and hist_b.last_epoch() == 11 and "param_groups" in state
    assert hist_b.pckh[-1]["val_pckh"] == 0.25 and hist_b.loss[-1]["val_loss"] == 0.6 and hist_b.best_pckh == 0.25
    for k, v in b.state_dict().items():
        assert torch.equal(v, a.state_dict()[k]), k


def test_lr_schedule_matches_reference(golden_dir):
    """cu-net.py::adjust_lr == utils/util.py:106-119 (x0.2 at epoch 101, x0.5 at 141 and 161), as the reference computed it."""
    import importlib.util
    import types
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("cu_net_entry", os.path.join(root, "cu-net.py"))
    entry = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(entry)
    ours = types.SimpleNamespace(lr=2.5e-4)
    lrs = [entry.adjust_lr(ours, e) for e in range(200)]
    assert lrs[100] == 2.5e-4 and abs(lrs[101] - 5e-5) < 1e-18 and abs(lrs[141] - 2.5e-5) < 1e-18 \
        and abs(lrs[199] - 1.25e-5) < 1e-18
    assert lrs == _reference(golden_dir)["adjust_lr"]


def test_quantizer_target_convs_match_reference_module_order(golden_dir):
    """QuanOp / BinOp pick nn.Conv2d modules by their modules()-index (utils/quantize.py:80-102): the parameter tree
    must enumerate its convs in the reference's order (features, hg, linears, intermedia -- models/cu_net.py:299-320)."""
    import torch.nn as nn
    from cunet_b200.models.cu_net import create_cu_net
    ours = create_cu_net(4, 32, 128, 5, 3, 2, 3)
    convs = [(n, tuple(m.weight.shape)) for n, m in ours.named_modules() if isinstance(m, nn.Conv2d)]
    assert convs == _reference(golden_dir)["convs_C5_L3_K2_loss3"] and len(convs) > 10
    assert convs[0][0] == "features.conv0" and convs[-1][0].startswith("intermedia.adapters.")
