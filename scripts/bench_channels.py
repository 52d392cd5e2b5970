import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np, torch
from helpers import synthetic_chain
from oracle import stitcher_ref
dev = torch.device('cuda', 0)
for c in (1, 3, 4):
    st, states, labels, images = synthetic_chain(6, 1080, 1920, c, kind='smooth')
    F = 32
    batch = {l: torch.from_numpy(np.stack([images[l]] * F)).to(dev) for l in labels}
    plan = st.plan([images[l].shape for l in labels], dev)
    out = plan.new_output(F, pitch_align=128)
    st.stitch_batch(batch, out=out); torch.cuda.synchronize()
    ref = stitcher_ref.stitch_chain(states, labels, images)
    ok = np.array_equal(out[0].cpu().numpy(), ref)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3): st.stitch_batch(batch, out=out)
    e0.record()
    for _ in range(10): st.stitch_batch(batch, out=out)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    ab = plan.algorithmic_bytes()
    print('C=%d exact=%s variant=%d ms=%.3f GB/s=%.0f frac=%.3f' % (c, ok, plan.handle.last_variant(), ms, ab * F / ms / 1e6, ab * F / ms / 1e6 / 6533.5))
