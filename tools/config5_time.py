import json, os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adafortitran_b200 import AdaFortiTranEstimator, ModelConfig, SystemConfig
from tests import util
sysc = SystemConfig(ofdm=dict(num_scs=3276, num_symbols=14), pilot=dict(num_scs=1638, num_symbols=2))
modc = ModelConfig(model_type="adafortitran", patch_size=(3, 2), num_layers=6, model_dim=128, num_head=4, activation="gelu",
                   max_seq_len=7644, pos_encoding_type="learnable", channel_adaptivity_hidden_sizes=[7, 42, 15288],
                   adaptive_token_length=6, device="cuda")
torch.manual_seed(0)
m = AdaFortiTranEstimator(sysc, modc).eval(); m.precision = "bf16"
B = int(sys.argv[1])
g = torch.Generator().manual_seed(3)
x = torch.complex(torch.randn(B, 1638, 2, generator=g), torch.randn(B, 1638, 2, generator=g)).cuda()
md = tuple(t.cuda() if torch.is_tensor(t) else t for t in util.meta(np.full(B, 20.0, np.float32), np.full(B, 50.0, np.float32), np.full(B, 500.0, np.float32)))
with torch.no_grad():
    m(x, md); torch.cuda.synchronize()
    for i in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter(); e0.record(); y = m(x, md); e1.record(); t1 = time.perf_counter(); torch.cuda.synchronize(); t2 = time.perf_counter()
        print(f"B={B} call {i}: device {e0.elapsed_time(e1):.2f} ms, host enqueue {1e3*(t1-t0):.2f} ms, total {1e3*(t2-t0):.2f} ms", flush=True)
