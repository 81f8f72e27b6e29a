"""Device time of the bit-rate kernel: training mode (noise buffer / in-kernel noise) and validation mode, at the image
table (374 612 rows) and the NeRF table (6 098 925 rows)."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from shacira_b200 import _lib  # noqa: E402

dev = torch.device("cuda", 0)
out = {}
for name, T, L in (("image", 374612, 16), ("nerf", 6098925, 16), ("nerf_total_only", 6098925, 0)):
    torch.manual_seed(0)
    w = torch.randn(T, 1, device=dev) * 6
    noise = torch.rand(T, 1, device=dev) - 0.5
    prob = torch.randn(4, 3, 1, device=dev) * 0.3
    first = [int(v) for v in torch.linspace(0, T, L + 1)[:-1]] if L else None
    def graphed(fn, reps=20):
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            fn()
            st.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                for _ in range(reps):
                    fn()
            g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            st.synchronize()
        return e0.elapsed_time(e1) / reps * 1e3

    out[name + "_train_us"] = graphed(lambda: _lib.entropy_bits(w, noise, prob, 2, first))
    out[name + "_val_us"] = graphed(lambda: _lib.entropy_bits(w, None, prob, 2, first, want_latent_grads=False))
print(json.dumps(out))
