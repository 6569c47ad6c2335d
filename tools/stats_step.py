"""Development: the config-2 launch and a 512-clip ragged statistics-only launch, timed for one build (ACB_LIB = the path of
another build of the library, default the in-tree library)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import audio_calm_b200 as acb
from bench import stats_clip_set, synth_batch
if os.environ.get("ACB_LIB"):
    acb._lib.LIB_PATH = os.environ["ACB_LIB"]
fe = acb.LogMelFrontend("cuda")
dev = torch.device("cuda")
lengths, starts, pool_len = stats_clip_set(2048)
pool = synth_batch(1, pool_len, "cuda", seed=99)[0]
b = acb.RaggedBatch(pool, torch.from_numpy(starts[:512]).to(dev), torch.from_numpy(lengths[:512]).to(dev), lengths[:512])
acc = acb.MelStatsAccumulator(80, "cuda")
peaks = fe.peak_abs_ragged(b)
x = synth_batch(256, 480000, "cuda")
out = torch.empty((256, 80, 1876), device="cuda")
aff = (acb.MEL_MEAN_DEFAULT, acb.MEL_STD_DEFAULT)
def timed(fn, n):
    for _ in range(5): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
t_plain = timed(lambda: fe.forward(x, affine=aff, out=out), 100)
t_stats = timed(lambda: fe.forward_ragged(b, pad_multiple=4, peak=peaks, moments=acc, stats_only=True), 100)
t_mom = timed(lambda: fe.forward(x, affine=aff, out=out, moments=acc), 100)
print(os.path.basename(os.environ.get("ACB_LIB", "in-tree")), "plain %.4f  ragged stats-only %.4f  uniform features+moments %.4f ms" % (t_plain, t_stats, t_mom), float(out.double().sum()))
