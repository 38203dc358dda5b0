"""Device time per kernel of the cfg-2 sampling step as the loop runs it (captured graph, replayed T times), padded and packed.

    python scripts/loop_kernel_profile.py [T]        # library: SEQDIFF_LIB, else the product build

torch.profiler (CUDA activities) around one T-step sampling after two warm-up samplings; kernels are grouped by name without
template arguments.  Prints one JSON object: per mode the library's launch count of a sampling, the device time per step and
per kernel name the time, launches and share per step.  The library's own event profiler marks only eager launches, so it
sees the stand-alone forward, not the loop's step."""
import json
import os
import re
import sys

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import seqdiff_b200 as sd  # noqa: E402

dev = torch.device("cuda:0")
torch.cuda.set_device(dev)
wl = bench.WORKLOADS["cfg2"]
bench.L = wl["L"]
B, T = wl["batch"], int(sys.argv[1]) if len(sys.argv) > 1 else 50
torch.manual_seed(0)
common = dict(max_position_embeddings=wl["L"], intermediate_size=bench.I, num_hidden_layers=bench.NL, position_embedding_type="relative_key")
model = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 20)
model = model.eval().to(dev)
model.precision = "bf16"
sched, trans = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20, timestep=500)
batch, x_T = bench.synthetic_workload(B, n_lig=wl["n_lig"], n_rec=wl["n_rec"])
db = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in batch.items()}
xT = x_T.to(dev)
out = {"lib": os.path.basename(sd._cabi.LIB_PATH), "T": T}
for packed in (False, True):
    def run():
        return sd.denoise_tensors(db, model, sched, trans, True, timesteps=T, x_T=xT, seed=5, graph_id0=0, packed=packed)
    run()
    run()
    torch.cuda.synchronize()
    n0 = sd.lib().seqdiff_launch_count()
    run()
    torch.cuda.synchronize()
    launches = sd.lib().seqdiff_launch_count() - n0
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        run()
        torch.cuda.synchronize()
    agg = {}
    for k in p.key_averages():
        us = getattr(k, "device_time_total", None)
        if us is None:
            us = k.cuda_time_total
        if not us:
            continue
        name = re.sub(r"^void ", "", k.key)
        name = re.sub(r"^seqdiff::(\(anonymous namespace\)::)?", "", name)
        name = re.split(r"[<(]", name)[0]
        a = agg.setdefault(name, [0.0, 0])
        a[0] += us
        a[1] += k.count
    tot = sum(v[0] for v in agg.values())
    out["packed" if packed else "padded"] = {
        "launches_per_sampling": launches, "us_per_step": round(tot / T, 1),
        "kernels": {n: {"us_per_step": round(v[0] / T, 2), "launches_per_step": round(v[1] / T, 2), "share": round(v[0] / tot, 4)}
                    for n, v in sorted(agg.items(), key=lambda kv: -kv[1][0])}}
print(json.dumps(out, indent=1))
