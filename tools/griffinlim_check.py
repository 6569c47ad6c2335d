import numpy as np, torch, sys
import os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import audio_calm_b200 as _acb
if os.environ.get("ACB_LIB"):
    _acb._lib.LIB_PATH = os.environ["ACB_LIB"]
from audio_calm_b200 import spectral
from oracle import spectral_oracle as so
g=np.load(os.path.join(ROOT, 'tests', 'golden', 'griffinlim_cases.npz'))
init=torch.from_numpy(g["init_angles"]).cuda(); mag=torch.from_numpy(g["mag"]).cuda()
for n in (2,8,32):
    w=spectral.griffin_lim(mag,n_iter=n,init_angles=init).cpu().numpy()
    o=so.griffin_lim(g["mag"][0],g["init_angles"][0],n_iter=n)
    line=f"n_iter {n}: gpu vs oracle {np.abs(w[0]-o).max()/np.abs(o).max():.2e}"
    if f"wave_{n}" in g: line+=f"  gpu vs torchaudio {np.abs(w-g[f'wave_{n}']).max()/np.abs(g[f'wave_{n}']).max():.2e}  oracle vs torchaudio {np.abs(o-g[f'wave_{n}'][0]).max()/np.abs(g[f'wave_{n}']).max():.2e}"
    print(line)
import time
x=torch.rand(8,513,626,device="cuda")+0.01
torch.cuda.synchronize(); t=time.perf_counter(); y=spectral.griffin_lim(x); torch.cuda.synchronize(); print("8 x 10 s clips, 32 iterations:", time.perf_counter()-t, "s")
import torchaudio
gl=torchaudio.transforms.GriffinLim(n_fft=1024).cuda()
gl(x); torch.cuda.synchronize(); t=time.perf_counter(); y2=gl(x); torch.cuda.synchronize(); print("torchaudio GriffinLim on the same GPU:", time.perf_counter()-t, "s")
t=time.perf_counter(); y=spectral.griffin_lim(x); torch.cuda.synchronize(); print("ours again:", time.perf_counter()-t, "s")
# per-kernel time of one iteration's launches
lib = __import__("audio_calm_b200")._lib.load()
spec = torch.randn(8, 513, 626, dtype=torch.complex64, device="cuda"); prev = torch.zeros_like(spec); magr = torch.rand(8, 513, 626, device="cuda")
wave = torch.empty(8, 512 * 625, device="cuda"); w = spectral._window(1024, wave.device); st = torch.cuda.current_stream().cuda_stream
def timed(fn, n=20):
    fn(); torch.cuda.synchronize(); e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True); e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize(); return e0.elapsed_time(e1) / n
print("istft (memset + kernel + normalise) ms:", timed(lambda: lib.acb_istft(spec.data_ptr(), 8, 626, 1024, 512, w.data_ptr(), wave.data_ptr(), 512 * 625, st)))
print("stft_complex + phase update ms:", timed(lambda: lib.acb_stft_complex(wave.data_ptr(), 8, 512 * 625, 1024, 512, w.data_ptr(), spec.data_ptr(), prev.data_ptr(), magr.data_ptr(), 0.497, st)))
wt = torch.hann_window(1024, device="cuda")
print("torch.istft ms:", timed(lambda: torch.istft(spec, 1024, 512, 1024, wt, length=512 * 625)), " torch.stft ms:", timed(lambda: torch.stft(wave, 1024, 512, 1024, wt, center=True, return_complex=True)))
print("stft_complex plain ms:", timed(lambda: lib.acb_stft_complex(wave.data_ptr(), 8, 512 * 625, 1024, 512, w.data_ptr(), spec.data_ptr(), None, None, 0.0, st)))
w256 = spectral._window(256, wave.device)
spec256 = torch.empty(8, 129, 1 + 320000 // 64, dtype=torch.complex64, device="cuda")
print("stft_complex n_fft 256 hop 64 ms:", timed(lambda: lib.acb_stft_complex(wave.data_ptr(), 8, 512 * 625, 256, 64, w256.data_ptr(), spec256.data_ptr(), None, None, 0.0, st)))
