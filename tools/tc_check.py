"""GPU scratch check of the tcgen05 path: self-tests, then bf16 forward vs oracle."""
import ctypes as C, json, os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adafortitran_b200 import _capi
from oracle import aft_oracle as O
from tests import util

def selftests():
    torch.cuda.init(); torch.zeros(1, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for which in (0, 1, 2, 4):
        err = C.c_double(-1)
        rc = _capi.lib().aft_selftest(which, C.byref(err), C.c_void_p(st))
        print(json.dumps({"selftest": which, "rc": rc, "max_err": err.value, "msg": _capi.lib().aft_last_error().decode()}), flush=True)

def forward_check(kind="ada", B=8):
    sd = util.ada_weights()
    if kind != "ada": sd = util.forti_weights(sd)
    p, snr, ds, dop = O.synthetic_batch(B, seed=3)
    ref = O.forward(util.oracle_cfg(kind), sd, p, snr, ds, dop)
    m = util.make_model(kind, weights=sd, precision="bf16")
    md = util.meta(snr, ds, dop) if kind == "ada" else None
    with torch.no_grad():
        y = m(torch.from_numpy(p), md)
    torch.cuda.synchronize()
    y = y.cpu().numpy()
    print(json.dumps({"bf16_forward": kind, "B": B, "normwise": O.normwise_err(y, ref), "rel_db": O.rel_err_db(y, ref),
                      "finite": bool(np.isfinite(y.view(np.float32)).all())}), flush=True)

def arm_diag():
    torch.zeros(1, device="cuda")
    err = C.c_double(-1)
    _capi.lib().aft_selftest(100, C.byref(err), None)

def dump_diag():
    err = C.c_double(-1)
    _capi.lib().aft_selftest(101, C.byref(err), None)
    print("diag records:", err.value, flush=True)

if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what == "timeline":
        sd = util.forti_weights(util.ada_weights())
        m = util.make_model("forti", weights=sd, precision="bf16")
        p, *_ = O.synthetic_batch(148 * 2, seed=3)      # 592 sequences: 4 per CTA
        tp = torch.from_numpy(p).cuda()
        with torch.no_grad():
            m(tp); torch.cuda.synchronize()
            err = C.c_double(-1)
            _capi.lib().aft_selftest(102, C.byref(err), None)
            m(tp); torch.cuda.synchronize()
            _capi.lib().aft_selftest(103, C.byref(err), None)
        print("timeline events:", err.value)
        sys.exit(0)
    if what == "diag":
        arm_diag()
        try:
            forward_check("forti", int(os.environ.get("AFT_DIAG_BATCH", "2")))
        except Exception as e:
            print("forward failed:", str(e)[:200])
        dump_diag()
        sys.exit(0)
    if what in ("all", "self"): selftests()
    if what in ("all", "fwd"):
        forward_check("forti", 2); forward_check("forti", 160); forward_check("ada", 8)
