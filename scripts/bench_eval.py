"""Validation-pass and prediction throughput (SURVEY.md §8f row 2; DESIGN.md §7.2, §7.3): ranking_metrics and predict() over a synthetic
frame at the c5 model size, wall clock per pass with a final device synchronise, and the share of the device-side kernels.  The reference
runs one forward per group and sorts on the host; the figure it would be compared with is groups/s of that loop (CPU oracle:
bench.py --impl reference).  The three passes alternate in one process so that they see the same clocks and the same neighbours."""
import os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from reactranker_b200 import _lib, synthetic
from reactranker_b200.data.load_reactions import DataProcessor, Parsing_features
from reactranker_b200.models.base_model import build_model
from reactranker_b200.predict import predict
from reactranker_b200.train import eval as E

G, N = (int(x) for x in (sys.argv[1] if len(sys.argv) > 1 else "410,50").split(","))
MC = 16
_lib.require_device(0)
ds = synthetic.make_dataset(7, [N] * G)
fz = Parsing_features(ds.mols)
df = ds.to_dataframe()
dp = DataProcessor(df)
torch.manual_seed(0)
model = build_model(hidden_size=300, mpnn_depth=3, mpnn_diff_depth=3, ffn_depth=3, use_bias=True, dropout=0.1, task_num=1,
                    ffn_last_layer="with_softplus", add_features_dim=1).cuda(0)
kw = dict(smiles_list=["rsmi_mapped", "psmi_mapped"], add_features_name="temp")
legs = {"ranking_metrics": lambda: E.ranking_metrics(model, 0, dp, fz, show_info=False, target_name="lgk", **kw),
        "predict mc_samples=1": lambda: predict(model, df, fz, 0, **kw),
        f"predict mc_samples={MC}": lambda: predict(model, df, fz, 0, mc_samples=MC, **kw)}
times = {k: [] for k in legs}
first = {}
for it in range(8):
    for name, fn in legs.items():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        times[name].append(time.perf_counter() - t0)
        if name == "ranking_metrics":
            metrics = r
ms = {k: np.median(v[2:]) * 1e3 for k, v in times.items()}
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
except OSError:
    card = torch.cuda.get_device_name(0)
print(f"device: {card}")
for k in legs:
    print(f"{k}: {G} groups x {N} candidates, median {ms[k]:.1f} ms per pass (spread {min(times[k][2:]) * 1e3:.1f}-{max(times[k][2:]) * 1e3:.1f}, "
          f"first {times[k][0] * 1e3:.0f} ms incl. store upload) = {G * N / ms[k] * 1e3:,.0f} reactions/s")
print(f"predict mc_samples=1 / ranking_metrics = {ms['predict mc_samples=1'] / ms['ranking_metrics']:.3f}; metrics {metrics[0]:.3f} {metrics[1]:.3f} "
      f"{metrics[2]:.3f} {np.round(metrics[3], 3)}")


def event_us(fn, reps=20):
    for _ in range(3):
        fn()
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return a.elapsed_time(e) / reps * 1e3


# the metrics kernel alone on the same shapes
scores = torch.randn(G * N, device="cuda:0")
t = np.random.default_rng(0).normal(size=G * N)
print(f"group_metrics (upload of targets + rr_rank_metrics): {event_us(lambda: E.group_metrics(scores, [N] * G, t)):.0f} us per call")
# rr_rank_predict alone on predict()'s launch shapes: GROUPS_PER_LAUNCH groups per call, T samples of one score column
L = _lib.lib()
for T in (1, MC):
    total = 0.0
    for lo in range(0, G, E.GROUPS_PER_LAUNCH):
        g = min(E.GROUPS_PER_LAUNCH, G - lo)
        s = torch.randn(T, g * N, device="cuda:0")
        off = torch.arange(0, (g + 1) * N, N, dtype=torch.int32, device="cuda:0")
        out = torch.empty(g * N, 6, device="cuda:0")
        total += event_us(lambda: _lib.check(L.rr_rank_predict(g * N, g, T, s.data_ptr(), g * N, 1, off.data_ptr(), N, out.data_ptr(), _lib.stream_ptr())))
    key = "predict mc_samples=1" if T == 1 else f"predict mc_samples={MC}"
    print(f"rr_rank_predict T={T}: {total:.1f} us per pass ({total / 1e3 / ms[key] * 100:.2f} % of a predict mc_samples={T} pass)")
