"""CPU: the training path's reference (Philox mask rule, fp64 restatement) and the plumbing of ``trainable``."""
import os
import re

import numpy as np
import pytest
import torch

from oracle import train_ref as T
from oracle.torch_port import TorchPort
from tests import util


def test_philox_known_answers():
    cases = [([0, 0, 0, 0], (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
             ([0xFFFFFFFF] * 4, (0xFFFFFFFF, 0xFFFFFFFF), "408f276d 41c83b0e a20bc7c6 6d5451fd"),
             ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], (0xA4093822, 0x299F31D0),
              "d16cfe09 94fdcceb 5001e420 24126ea1")]
    for ctr, key, want in cases:
        got = T.philox4x32_10([np.array([c], dtype=np.uint32) for c in ctr], key)
        assert " ".join(f"{int(w[0]):08x}" for w in got) == want


def test_keep_rate_and_independence():
    m = T.keep_mask(0x1234_5678_9ABC, 3, 2, 1, (1000, 1000), 0.1)
    assert abs(m.mean() - 0.9) < 0.002
    other = T.keep_mask(0x1234_5678_9ABC, 4, 2, 1, (1000, 1000), 0.1)    # the imaginary pass of the same sample
    assert (m != other).mean() > 0.1
    assert T.keep_mask(5, 0, 0, 0, (4, 280, 280), 0.0).all()


def _grads(out, params, g):
    loss = (out * g).sum()
    return torch.autograd.grad(loss, params, allow_unused=True)


@pytest.mark.parametrize("kind", ["ada", "forti"])
def test_restatement_matches_torch_port(kind):
    sd = util.ada_weights() if kind == "ada" else util.forti_weights(util.ada_weights())
    adaptive = kind == "ada"
    port = TorchPort(sd, adaptive=adaptive, num_layers=6).double()
    port.eval()
    P = {k: v.double().requires_grad_(True) for k, v in T.params_from_state_dict(sd, adaptive, 6).items()}
    rng = np.random.default_rng(0)
    n = 2
    x = torch.from_numpy(rng.standard_normal((n, 24)))
    cond = [torch.tensor([[v], [v + 3.0]], dtype=torch.float64) for v in (10.0, 50.0, 300.0)] if adaptive else None
    ones = [[torch.ones(n, *T.SITE_SHAPES[s], dtype=torch.float64) for s in range(4)] for _ in range(6)]
    ours = T.real_pass(P, x, cond, ones, 0.0, 6)
    with torch.enable_grad():
        ref = port._real(x, cond)
    assert torch.allclose(ours, ref, rtol=0, atol=1e-12 * float(ref.detach().abs().max()))
    g = torch.from_numpy(rng.standard_normal(ref.shape))
    ref_params = dict(port.named_parameters())
    gp = _grads(ours, list(P.values()), g)
    gr = torch.autograd.grad((ref * g).sum(), list(ref_params.values()))
    gr = dict(zip(ref_params, gr))
    # map a few representative tensors of every part of the model
    pairs = {"up_w": "up.weight", "enh_w1": "enh.2.weight", "ref_b3": "ref.6.bias", "l1_w": "l1.weight",
             "l2_w": "l2.weight", "L0_in_w": "enc.layers.0.self_attn.in_proj_weight",
             "L5_n2_w": "enc.layers.5.norm2.weight", "L3_l1_b": "enc.layers.3.linear1.bias"}
    if adaptive:
        pairs.update(snr_w0="mlps.0.0.weight", dop_w2="mlps.2.4.weight")
    names = list(P)
    for ours_name, ref_name in pairs.items():
        a, b = gp[names.index(ours_name)], gr[ref_name]
        assert torch.linalg.norm(a - b) <= 1e-12 * torch.linalg.norm(b), ours_name
    # rows of the positional table beyond the 280 tokens receive no gradient
    assert gp[names.index("pos")][0, 280:].abs().max() == 0


def test_trainable_plumbing_on_cpu_model():
    a = util.make_model("ada", device="cpu")
    md = util.meta([0, 0], [50, 50], [200, 200])
    x = torch.zeros(2, 12, 2, dtype=torch.cfloat)
    assert a.trainable is False
    a.train()
    with pytest.raises(RuntimeError, match="inference-only"):
        a(x, md)
    a.trainable = True
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        a(x, md)
    a.precision = "bf16"
    with pytest.raises(ValueError, match="fp32"):
        a(x, md)
    a.precision = "fp32"
    with pytest.raises(ValueError, match="gather"):
        a(x, md, gather=object())
    with pytest.raises(ValueError, match="pilots or the metadata"):
        a(x.clone().requires_grad_(True), md)
    with pytest.raises(RuntimeError, match="forward_host is inference-only"):
        a.forward_host(x, md)
    a.eval()                                   # eval mode with grad enabled is still a differentiable call
    with pytest.raises(RuntimeError, match="forward_host is inference-only"):
        a.forward_host(x, md)
    with torch.no_grad():                      # no grad: the inference path, which refuses a CPU model as before
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            a(x, md)


def test_training_exports_in_header():
    header = open(os.path.join(util.ROOT, "include", "aft.h")).read()
    declared = set(re.findall(r"AFT_API\s+[\w\s\*]+?\b(aft_\w+)\s*\(", header))
    assert {"aft_param_count", "aft_train_workspace_bytes", "aft_forward_train", "aft_backward"} <= declared
    assert re.search(r"#define AFT_ABI_VERSION 3\b", header)
