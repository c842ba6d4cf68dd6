"""GPU: the fp32 training path (aft_forward_train / aft_backward behind autograd) against the fp64 restatement of
``oracle/train_ref.py``.

Errors are normwise, ||x - x64|| / ||x64||.  Outputs are gated at 1e-4.  Gradients and parameter updates are gated
against what stock fp32 autograd reaches on the same restatement, inputs and masks (the "stock" arm, on the CPU): a few
gradients are out of reach of any fp32 implementation at 1e-4 -- relu' changes sign between fp32 and fp64 for
pre-activations near zero, and some bias-like gradients are sums whose terms largely cancel -- so each tensor, and the
concatenation of all of them, must be within K times the stock fp32 error, or within 1e-4."""
import numpy as np
import pytest
import torch

from oracle import aft_oracle as O
from oracle import train_ref as T
from tests import util

pytestmark = pytest.mark.gpu
TOL = 1e-4
K = 4.0


def _inputs(n, seed):
    rng = np.random.default_rng(seed)
    pilots, snr, ds, dop = O.synthetic_batch(n, seed=seed)
    g = (rng.standard_normal((n, 120, 14)) + 1j * rng.standard_normal((n, 120, 14))).astype(np.complex128)
    return pilots, (snr, ds, dop), g


def _nw(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    den = np.linalg.norm(b)
    return np.linalg.norm(a - b) / den if den > 0 else np.linalg.norm(a)


def _run_ours(model, pilots, cond, g=None, truth=None, torch_seed=0):
    """One differentiable call: returns (out, {name: grad or None}); loss = <g, out> or the reference MSE."""
    model.zero_grad(set_to_none=True)
    md = util.meta(*cond) if model.use_channel_adaptation else None
    torch.manual_seed(torch_seed)
    out = model(torch.from_numpy(pilots), md)
    if g is not None:
        gt = torch.from_numpy(g).to(out.device)
        loss = (out.real * gt.real.float() + out.imag * gt.imag.float()).sum()
    else:
        t = torch.from_numpy(truth).to(out.device)
        loss = torch.nn.functional.mse_loss(torch.cat([out.real, out.imag], 1), torch.cat([t.real, t.imag], 1))
    loss.backward()
    named, _ = model._weight_tensors()
    return out.detach().cpu().numpy(), {n: (None if t.grad is None else t.grad.detach().cpu().numpy()) for n, t in named}


def _run_ref(model, pilots, cond, p, seed, g=None, truth=None, dtype=torch.float64, masks=None):
    """The restatement on the CPU in ``dtype`` (fp64: the reference; fp32: stock fp32 autograd)."""
    named, _ = model._weight_tensors()
    P = {n: t.detach().cpu().to(dtype).requires_grad_(True) for n, t in named}
    mc = model.model_config
    c = [np.asarray(v, np.float64) for v in cond] if model.use_channel_adaptation else None
    ctype = torch.complex128 if dtype == torch.float64 else torch.complex64
    out = T.forward(P, torch.from_numpy(pilots).to(ctype), c, p, seed, mc.num_layers, mc.activation, masks=masks)
    if g is not None:
        gt = torch.from_numpy(g).to(ctype)
        loss = (out.real * gt.real + out.imag * gt.imag).sum()
    else:
        t = torch.from_numpy(truth).to(ctype)
        loss = torch.nn.functional.mse_loss(torch.cat([out.real, out.imag], 1), torch.cat([t.real, t.imag], 1))
    grads = torch.autograd.grad(loss, list(P.values()))
    return out.detach().numpy(), {n: gr.double().numpy() for n, gr in zip(P, grads)}


def _gate(ours, stock, ref, what):
    """ours / stock / ref: {name: array}.  Each tensor and the concatenation within max(TOL, K * stock error)."""
    rows = []
    for n in ref:
        e, es = _nw(ours[n], ref[n]), _nw(stock[n], ref[n])
        rows.append((n, e, es))
    cat = lambda d: np.concatenate([np.asarray(d[n], np.float64).ravel() for n in ref])
    e_all, es_all = _nw(cat(ours), cat(ref)), _nw(cat(stock), cat(ref))
    worst = sorted(rows, key=lambda r: -r[1])[:4]
    print(f"{what}: all {e_all:.2e} (stock fp32 {es_all:.2e}); worst tensors",
          ", ".join(f"{n} {e:.2e} (stock {es:.2e})" for n, e, es in worst))
    bad = [(n, e, es) for n, e, es in rows if e > max(TOL, K * es)]
    assert not bad, (what, bad)
    assert e_all <= max(TOL, K * es_all), (what, e_all, es_all)


def _seed_of(torch_seed):
    torch.manual_seed(torch_seed)
    return int(torch.randint(0, 2 ** 62, (), dtype=torch.int64).item())


def _check_grads(ours, ref, stock, what, sinusoidal=False):
    if sinusoidal:
        assert ours["pos"] is None
        ours, ref, stock = ({n: v for n, v in d.items() if n != "pos"} for d in (ours, ref, stock))
    else:
        assert np.all(ours["pos"][0, 280:] == 0)
    assert all(g is not None for g in ours.values())
    _gate(ours, stock, ref, what)


def _trained_sd():
    t = util.golden("golden_trained.npz")
    return {k[3:]: v for k, v in t.items() if k.startswith("sd/")}


CASES = {
    "ada_trained": dict(kind="ada", n=3, weights=lambda sd: _trained_sd()),
    "forti_seed0": dict(kind="forti", n=4, weights=util.forti_weights),
    "relu": dict(kind="ada", n=2, overrides={"activation": "relu"}),
    "layers2": dict(kind="ada", n=2, overrides={"num_layers": 2},
                    weights=lambda sd: {k: a for k, a in sd.items() if not any(f"layers.{i}." in k for i in range(2, 6))}),
    "sinusoidal": dict(kind="ada", n=2, overrides={"pos_encoding_type": "sinusoidal"},
                       weights=lambda sd: {k: a for k, a in sd.items() if "position_embeddings" not in k}),
}


def _case_model(name):
    c = CASES[name]
    sd = util.ada_weights()
    w = c.get("weights", lambda s: s)(sd)
    if c.get("overrides", {}).get("pos_encoding_type") == "sinusoidal":
        m = util.make_model(c["kind"], overrides=c.get("overrides"))
        own = m.state_dict()
        w = dict(w, **{"transformer_encoder.positional_encoding.pe": own["transformer_encoder.positional_encoding.pe"].cpu().numpy()})
        m.load_state_dict(util.to_torch(w))
    else:
        m = util.make_model(c["kind"], overrides=c.get("overrides"), weights=w)
    m.trainable = True
    return m.eval(), c["n"]


@pytest.mark.parametrize("case", list(CASES))
def test_gradients_p0(case):
    model, n = _case_model(case)
    pilots, cond, g = _inputs(n, seed=11)
    sin = case == "sinusoidal"
    out, ours = _run_ours(model, pilots, cond, g=g)
    ref_out, ref = _run_ref(model, pilots, cond, 0.0, None, g=g)
    _, stock = _run_ref(model, pilots, cond, 0.0, None, g=g, dtype=torch.float32)
    assert _nw(out.view(np.float32), ref_out.view(np.float64)) <= TOL
    _check_grads(ours, ref, stock, f"{case} <g, out>", sin)
    # the reference's loss: MSE over concatenated real / imaginary parts
    truth = O.synthetic_channel(n, 10.0, 100.0, 400.0, seed=3)[1]
    _, ours = _run_ours(model, pilots, cond, truth=truth)
    _, ref = _run_ref(model, pilots, cond, 0.0, None, truth=truth)
    _, stock = _run_ref(model, pilots, cond, 0.0, None, truth=truth, dtype=torch.float32)
    _check_grads(ours, ref, stock, f"{case} mse", sin)


def test_training_forward_p0_matches_inference():
    model, n = _case_model("ada_trained")
    pilots, cond, _ = _inputs(5, seed=2)
    md = util.meta(*cond)
    with torch.no_grad():
        inf = model(torch.from_numpy(pilots), md).cpu().numpy()
    tr = model(torch.from_numpy(pilots), md).detach().cpu().numpy()   # eval + grad enabled: training forward, p = 0
    assert _nw(tr.view(np.float32), inf.view(np.float32)) <= 1e-6


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_dropout_matches_restatement(p):
    model = util.make_model("ada", overrides={"dropout": p}, weights=util.ada_weights())
    model.trainable = True
    model.train()
    pilots, cond, g = _inputs(2, seed=5)
    out, ours = _run_ours(model, pilots, cond, g=g, torch_seed=123)
    masks = [T.masks_for(_seed_of(123), 2, e, 6, p) for e in (0, 1)]
    ref_out, ref = _run_ref(model, pilots, cond, p, None, g=g, masks=masks)
    _, stock = _run_ref(model, pilots, cond, p, None, g=g, dtype=torch.float32, masks=masks)
    assert _nw(out.view(np.float32), ref_out.view(np.float64)) <= TOL
    _check_grads(ours, ref, stock, f"dropout {p}")


def test_same_seed_bit_identical_other_seed_differs():
    model = util.make_model("ada", weights=util.ada_weights())
    model.trainable = True
    model.train()
    pilots, cond, g = _inputs(3, seed=6)
    o1, g1 = _run_ours(model, pilots, cond, g=g, torch_seed=7)
    o2, g2 = _run_ours(model, pilots, cond, g=g, torch_seed=7)
    assert np.array_equal(o1, o2)
    for n in g1:
        assert np.array_equal(g1[n], g2[n]), n
    o3, _ = _run_ours(model, pilots, cond, g=g, torch_seed=8)
    assert not np.array_equal(o1, o3)


def test_sgd_steps_match_fp64():
    """5 SGD steps (lr 1e-3, p = 0) from seed-0 weights on fixed batches: theta_5 - theta_0 of the model's own fp32
    parameters -- optimizer.step(), the repack the version counters trigger, the next training forward -- against the
    same steps in fp64, gated by the same steps in stock fp32 autograd (whose parameters round the same way)."""
    model = util.make_model("ada", weights=util.ada_weights())
    model.trainable = True
    named, _ = model._weight_tensors()
    theta0 = {n: t.detach().cpu().double().clone() for n, t in named}
    arms = {dt: {n: t.to(dt).clone().requires_grad_(True) for n, t in theta0.items()} for dt in (torch.float64, torch.float32)}
    opts = {dt: torch.optim.SGD(list(P.values()), lr=1e-3) for dt, P in arms.items()}
    opt = torch.optim.SGD(model.parameters(), lr=1e-3)
    mse = lambda o, t: torch.nn.functional.mse_loss(torch.cat([o.real, o.imag], 1), torch.cat([t.real, t.imag], 1))
    for step in range(5):
        pilots, h = O.synthetic_channel(2, 15.0, 100.0, 600.0, seed=100 + step)
        cond = (np.full(2, 15.0, np.float32), np.full(2, 100.0, np.float32), np.full(2, 600.0, np.float32))
        opt.zero_grad()
        out = model(torch.from_numpy(pilots), util.meta(*cond))
        mse(out, torch.from_numpy(h).to(out.device)).backward()
        opt.step()
        for dt, P in arms.items():
            ct = torch.complex128 if dt == torch.float64 else torch.complex64
            opts[dt].zero_grad()
            o = T.forward(P, torch.from_numpy(pilots).to(ct), [c.astype(np.float64) for c in cond], 0.0, None, 6)
            mse(o, torch.from_numpy(h).to(ct)).backward()
            opts[dt].step()
    named, _ = model._weight_tensors()
    ours = {n: (t.detach().cpu().double() - theta0[n]).numpy() for n, t in named}
    ref = {n: (arms[torch.float64][n].detach() - theta0[n]).numpy() for n in theta0}
    stock = {n: (arms[torch.float32][n].detach().double() - theta0[n]).numpy() for n in theta0}
    _gate(ours, stock, ref, "sgd theta_5 - theta_0")


def _recipe_batch(rng, n, seed):   # tests/golden/make_golden_trained.py: batch()
    snr = rng.choice(O.SNR_GRID, size=n).astype(np.float32)
    ds = rng.choice(O.DS_GRID, size=n).astype(np.float32)
    dop = rng.choice(O.DOP_GRID, size=n).astype(np.float32)
    ps, hs = [], []
    for i in range(n):
        p, h = O.synthetic_channel(1, float(snr[i]), float(ds[i]), float(dop[i]), seed=seed * 1000 + i)
        ps.append(p[0]), hs.append(h[0])
    return np.stack(ps), np.stack(hs), snr, ds, dop


def test_recipe_replay_reaches_reference_nmse():
    """The training recipe of make_golden_trained.py (Adam 5e-4, batch 32, clip 1.0, dropout 0.1, rng 7) for 150 steps.

    The reference's recorded trace sits at 0 dB until about step 50 and then drops (-4.0 dB over steps 100-125, -4.1 dB
    over 125-150).  When that drop happens is sensitive to rounding: this run is deterministic and reached -3.5 dB over
    steps 125-150 on a B200, while an earlier build that summed the small gradients in fp32 reached -2.1 dB."""
    torch.manual_seed(0)
    model = util.make_model("ada")
    model.trainable = True
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    rng = np.random.default_rng(7)
    trace = []
    for step in range(150):
        p, h, snr, ds, dop = _recipe_batch(rng, 32, step)
        est = model(torch.from_numpy(p), util.meta(snr, ds, dop))
        truth = torch.from_numpy(h).to(est.device)
        loss = torch.nn.functional.mse_loss(torch.cat([est.real, est.imag], 1), torch.cat([truth.real, truth.imag], 1))
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        trace.append(10 * np.log10(float((est - truth).abs().pow(2).sum() / truth.abs().pow(2).sum())))
    late = float(np.mean(trace[125:150]))
    print(f"recipe replay: mean training NMSE over steps 125-150 = {late:.2f} dB")
    assert np.isfinite(trace).all() and late <= -3.0


def test_error_paths():
    from adafortitran_b200 import FortiTranEstimator, ModelConfig, SystemConfig
    m = FortiTranEstimator(SystemConfig(ofdm=dict(num_scs=24, num_symbols=8), pilot=dict(num_scs=4, num_symbols=2)),
                           ModelConfig(**dict(util.FORTI, device="cuda")))
    m.trainable = True
    with pytest.raises(ValueError, match="default geometry"):
        m(torch.zeros(2, 4, 2, dtype=torch.complex64))
    model = util.make_model("ada", weights=util.ada_weights())
    model.trainable = True
    pilots, cond, _ = _inputs(2, seed=1)
    out = model(torch.from_numpy(pilots), util.meta(*cond))
    loss = out.abs().pow(2).sum()
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="second time"):
        loss.backward()
