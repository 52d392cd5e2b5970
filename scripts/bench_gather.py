import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np, torch
from helpers import synthetic_chain
dev = torch.device('cuda', 0)
st, states, labels, images = synthetic_chain(6, 1080, 1920, 3, kind='smooth')
F = 32
batch = {l: torch.from_numpy(np.stack([images[l]] * F)).to(dev) for l in labels}
plan = st.plan([images[l].shape for l in labels], dev)
out = plan.new_output(F, pitch_align=128)
for v, mode in ((2, ''), (1, ''), (1, 'MCS_GATHER_BYTES')):
    plan.handle.force_variant(v)
    os.environ.pop('MCS_GATHER_BYTES', None)
    if mode:
        os.environ[mode] = '1'   # read by the library at every call
    st.stitch_batch(batch, out=out); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3): st.stitch_batch(batch, out=out)
    e0.record()
    for _ in range(10): st.stitch_batch(batch, out=out)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    ab = plan.algorithmic_bytes()
    print('variant=%d mode=%s ms=%.3f frac=%.3f' % (plan.handle.last_variant(), mode, ms, ab * F / ms / 1e6 / 6533.5))
