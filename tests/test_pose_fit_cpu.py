"""CPU checks of pose fitting with a frozen field (training.PoseFitStep): every refusal is raised before anything is
set up, the render block and the graph net refuse a parameter set in which only some parameters need a gradient, and
the ctypes signatures of the entry points whose pose-only variants take NULL still match the header."""
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import danbo_b200                                    # noqa: E402,F401
from danbo_b200 import _lib, autograd, networks, pose_opt as po, training   # noqa: E402

FX = np.load(os.path.join(ROOT, "tests", "golden", "popt.npz"))


def _stand_in(graph_net=True, fine=False):
    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Parameter(torch.full((3,), 0.5))
            if graph_net:
                self.graph_net = torch.nn.Linear(1, 1)

    class Caster(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.network = Net()
            if fine:
                self.network_fine = Net()
    return Caster()


def _popt(**kw):
    args = types.SimpleNamespace(opt_rot6d=False, opt_pose_lrate=1e-2, init_poseopt=None, no_poseopt_reload=False,
                                 use_ckpt_anchor=False, opt_pose_cache=False, opt_pose_tol=0.0, opt_pose_coef=2.0,
                                 use_temp_loss=False, ext_scale=0.001, lrate=1e-2, loss_fn="L1", agg_type="sigmoid")
    for k, v in kw.items():
        setattr(args, k, v)
    attrs = {"rest_pose": FX["rest_pose"], "betas": np.zeros((1, 10), np.float32), "kp3d": FX["init_kps"],
             "bones": FX["init_bones"]}
    opt, popt = po.create_popt(args, attrs)
    return args, opt, popt


@pytest.mark.parametrize("case,word", [("anerf", "A-NeRF"), ("fine", "fine network"), ("world", "world_size"),
                                       ("rot6d", "opt_rot6d"), ("temp", "use_temp_loss"), ("cache", "opt_pose_cache"),
                                       ("adam", "FlatAdam")])
def test_pose_fit_refusals(case, word):
    args, opt, popt = _popt(opt_rot6d=case == "rot6d", use_temp_loss=case == "temp", opt_pose_cache=case == "cache")
    caster = _stand_in(graph_net=case != "anerf", fine=case == "fine")
    state = {k: v.clone() for k, v in caster.state_dict().items()}
    layer = {k: v.clone() for k, v in popt["popt_layer"].state_dict().items()}
    for graph in (False, True):
        with pytest.raises(NotImplementedError, match=f"pose fitting .*{word}"):
            training.PoseFitStep(caster, args, popt, opt, graph=graph, world_size=2 if case == "world" else 1)
    # refused before anything was set up: no gradient, no weight and no pose moved, nothing left on the caster
    assert all(p.grad is None for p in caster.parameters())
    assert all(torch.equal(v, state[k]) for k, v in caster.state_dict().items())
    assert all(torch.equal(v, layer[k]) for k, v in popt["popt_layer"].state_dict().items())
    assert not hasattr(caster, "grads_in_place")


def test_pose_fit_needs_a_pose_layer():
    args, opt, _ = _popt()
    with pytest.raises(ValueError, match="pose layer"):
        training.PoseFitStep(_stand_in(), args, {"popt_layer": None}, opt)


def test_pose_fit_refuses_batches_without_equal_runs():
    # the batch check is the first thing a call does (PoseFitStep needs a CUDA FlatAdam to be built, so the bare
    # object stands in: a call that got past the check would fail on the missing attributes instead)
    step = training.PoseFitStep.__new__(training.PoseFitStep)
    with pytest.raises(NotImplementedError, match="unique"):
        step({"kp_idx": torch.zeros(10, dtype=torch.long), "N_uniques": 4})


def test_weight_grads_decides_all_or_none():
    core = autograd.N_TRAINED
    n = len(autograd.PARAM_NAMES)
    assert autograd.weight_grads([True] * n, core) is True
    # axis_scale without opt_scale, the zero code table of a field without frame codes: constants beside a trained field
    assert autograd.weight_grads([True] * core + [False] * (n - core), core) is True
    assert autograd.weight_grads([False] * n, core) is False
    for flags in ([True] * (core - 1) + [False] * (n - core + 1), [False] * core + [True] * (n - core),
                  [False] + [True] * (n - 1)):
        with pytest.raises(NotImplementedError, match="only some"):
            autograd.weight_grads(flags, core)


def test_render_block_refuses_a_mixed_parameter_set():
    net = networks.DanboField()
    caster = types.SimpleNamespace(network=net)
    named = dict(net.named_parameters())
    named["pts_linears.3.weight"].requires_grad_(False)
    with pytest.raises(NotImplementedError, match="only some"):
        # refused before the node is built: none of the (here meaningless) render arguments is read
        autograd.render_block_with_grad(caster, None, 1, None, None, None, None, None, None, None, 8, 8, 1.0, 0., 0.,
                                        None, {}, None)
    for p in net.parameters():
        p.requires_grad_(False)
    named["prob_linears.layers.1.bias"].requires_grad_(True)
    with pytest.raises(NotImplementedError, match="only some"):
        autograd.render_block_with_grad(caster, None, 1, None, None, None, None, None, None, None, 8, 8, 1.0, 0., 0.,
                                        None, {}, None)


def test_graph_net_refuses_a_mixed_parameter_set():
    net = networks.DanboField()
    dict(net.graph_net.named_parameters())["layers.2.bias"].requires_grad_(False)
    pose = torch.zeros(2, 24, 3, requires_grad=True)
    with pytest.raises(NotImplementedError, match="only some"):
        autograd.graph_net_volumes(net, pose)


def _header_args(name):
    text = open(os.path.join(ROOT, "include", "danbo_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)", text)
    return [a.strip() for a in m.group(1).split(",")]


@pytest.mark.parametrize("name", ["danbo_mlp_dgrad", "danbo_mlp_head_bwd", "danbo_field_agg_bwd", "danbo_graph_net_bwd"])
def test_pose_only_entry_points_match_the_header(name):
    """The pose-only variants are selected by NULL pointers: the signatures, and so the ctypes table, are unchanged."""
    import ctypes
    args = _header_args(name)
    sig = _lib._SIGNATURES[name]
    assert len(sig) == len(args)
    for a, t in zip(args, sig):
        is_ptr = "*" in a
        assert (t is ctypes.c_void_p) == is_ptr, (name, a, t)
    assert _lib.ABI_VERSION == 5
