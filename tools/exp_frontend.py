"""Developer experiment (GPU box): front-end stage time (CUDA events of the library) and, with `trace` as the second argument,
the per-job timeline of the single-launch front end (fl_debug_option FL_OPT_TRACE)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import fealess_b200 as fb
from fealess_b200 import synth

W, H, T = 640, 480, (5, 8)
NT = int(sys.argv[1]) if len(sys.argv) > 1 else 8000
frames = [synth.make_frame(W, H, i) for i in range(4)]
h = fb.Handle(T, (0, 1), W, H)
TRACE = len(sys.argv) > 2 and sys.argv[2] == "trace"
if TRACE:
    h.debug_option(fb.FL_OPT_TRACE, 1)
h.upload_templates(synth.make_templates(0))
rc, _, q = h.match(frames[0][0], frames[0][1], 75.0, want_quantized=True)
ts = synth.make_templates(NT, W, H, T, seed=1, quantized=q, planted_fraction=0.01)
h.upload_templates(ts)
h.profile(True)
import ctypes as C
st = np.zeros(4); n = 0
tl = np.zeros(4)
tl2 = np.zeros(4)
cnt = np.zeros(16, np.int32)
for it in range(104):
    b, d = frames[it % 4]
    rc, m = h.match(b, d, 75.0)
    if it >= 4:
        st += h.last_stage_ms(); n += 1
        fb.lib().fl_debug_get(h._h, 5, 0, 0, 0, C.c_void_p(cnt.ctypes.data), C.c_size_t(cnt.nbytes))
        tl += cnt[8:12]
        tl2 += cnt[4:8]
        if it < 8:
            print("frame %d: unique %d live %d raw %d | sort body ns: counts %d gather %d sort %d output %d" % (it % 4, cnt[0], cnt[1], cnt[3], cnt[4], cnt[5], cnt[6], cnt[7]))
if TRACE:
    fe = h.fe_trace()
    if len(fe):
        t0 = fe[:, 2].min()
        names = {2: "pyrDown", 3: "resize", 4: "spread+LM", 5: "colour", 6: "depth", 7: "prefetch"}
        for k, c, a, b, _, _ in fe:
            print("FE job %-10s %5d CTAs: first start %6.2f us, last end %6.2f us" % (names.get(int(k), "?"), c, (a - t0) / 1e3, (b - t0) / 1e3))
st /= n
tl /= n
tl2 /= n
print("sort body (rank path) timeline, mean us: counts %.2f, gather %.2f, rank+scan %.2f, output %.2f" % tuple(tl2 / 1e3))
print("refine+sort kernel timeline (last CTA), mean: refine %.2f us, ticket %.2f us, sort %.2f us, candidates %.1f" % (tl[0] / 1e3, tl[1] / 1e3, tl[2] / 1e3, tl[3]))
print("matches %d | stage us: fe %.1f sim %.1f refine %.1f sort %.1f total %.1f"
      % (len(m), *(1e3 * st), 1e3 * st.sum()), flush=True)
