"""Device time per kernel of the cfg-2 sampling step as the loop runs it (captured graph, replayed T times), padded and packed.

    python scripts/loop_kernel_profile.py [T] [K]    # library: SEQDIFF_LIB, else the product build

torch.profiler (CUDA activities) around one T-step sampling after two warm-up samplings; kernels are grouped by name without
template arguments.  Prints one JSON object: per mode the library's launch count of a sampling, the device time per step and
per kernel name the time, launches and share per step.  The library's own event profiler marks only eager launches, so it
sees the stand-alone forward, not the loop's step.
K > 1: the workload's B graphs become B / K pockets x K samples, profiled both as the replicated batch ("<mode>_replicated",
seqdiff_sample_ex) and with the pockets shared ("<mode>_shared", seqdiff_sample_multi).  Every kernel of the step is also listed
by its position in the step ("by_position": the kernel trace cut at each reverse_step_kernel, mean device time over the full
steps), which tells apart launches of the same kernel, e.g. the cross K|V GEMM from the decoder's GEMMs."""
import json
import os
import re
import sys
import tempfile

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
K = int(sys.argv[2]) if len(sys.argv) > 2 else 1
torch.manual_seed(0)
common = dict(max_position_embeddings=wl["L"], intermediate_size=bench.I, num_hidden_layers=bench.NL, position_embedding_type="relative_key")
model = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 20)
model = model.eval().to(dev)
model.precision = "bf16"
sched, trans = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20, timestep=500)
batch, x_T = bench.synthetic_workload(B // K, n_lig=wl["n_lig"], n_rec=wl["n_rec"])
batch.pop("structure_ids")
db = {k: v.to(dev) for k, v in batch.items()}
xT = torch.nn.functional.one_hot(torch.randint(0, 20, (B, wl["L"]), generator=torch.Generator().manual_seed(4)), 20).float().to(dev) if K > 1 else x_T.to(dev)
out = {"lib": os.path.basename(sd._cabi.LIB_PATH), "T": T}
if K > 1:
    out["K"] = K
forms = [(False, ""), (True, "")] if K == 1 else [(p, f) for p in (False, True) for f in ("_replicated", "_shared")]
for packed, form in forms:
    def run():
        b = {k: v.repeat_interleave(K, dim=0) for k, v in db.items()} if form == "_replicated" else db
        return sd.denoise_tensors(b, model, sched, trans, True, timesteps=T, x_T=xT, seed=5, graph_id0=0, packed=packed,
                                  num_samples=K if form == "_shared" else 1)
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
    rec = out[("packed" if packed else "padded") + form] = {
        "launches_per_sampling": launches, "us_per_step": round(tot / T, 1),
        "kernels": {n: {"us_per_step": round(v[0] / T, 2), "launches_per_step": round(v[1] / T, 2), "share": round(v[0] / tot, 4)}
                    for n, v in sorted(agg.items(), key=lambda kv: -kv[1][0])}}
    with tempfile.TemporaryDirectory() as d:
        p.export_chrome_trace(os.path.join(d, "trace.json"))
        events = json.load(open(os.path.join(d, "trace.json")))["traceEvents"]
    kern = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    cuts = [i for i, e in enumerate(kern) if "reverse_step_kernel" in e["name"]]
    steps = [kern[a + 1:b + 1] for a, b in zip(cuts, cuts[1:])]  # full steps: after one reverse step up to the next
    n = len(steps[0])
    assert all(len(st) == n for st in steps), "steps of different kernel counts"
    rec["by_position"] = [{"kernel": re.split(r"[<(]", re.sub(r"^(void )?seqdiff::", "", steps[0][i]["name"]))[0],
                           "grid": steps[0][i]["args"]["grid"], "us": round(sum(st[i]["dur"] for st in steps) / len(steps), 2)}
                          for i in range(n)]
print(json.dumps(out, indent=1))
