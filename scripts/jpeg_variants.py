"""Decode time of 32 x 24 MP streams for library variants (CUDA events, best of 3): WITHOUT restart markers, or with a restart
interval of JV_RI MCUs when that environment variable is set."""
import io, os, subprocess, sys
CHILD = r'''
import io, os, sys
import numpy as np, torch
from PIL import Image
sys.path.insert(0, ".")
from facet_b200 import ops
from facet_b200.synth import synth_image_bgr
from facet_b200.utils import jpeg as fj
H, W, n = 4000, 6000, 32
datas = []
for i in range(2):
    buf = io.BytesIO()
    kw = {"restart_marker_blocks": int(os.environ["JV_RI"])} if os.environ.get("JV_RI") else {}
    Image.fromarray(synth_image_bgr(2000 + i, H, W)[:, :, ::-1].copy()).save(buf, "JPEG", quality=90, **kw)
    datas.append(np.frombuffer(buf.getvalue(), np.uint8).copy())
streams = [datas[i % 2] for i in range(n)]
infos = [fj.parse(s) for s in streams]
slot = (max(len(s) for s in streams) + 255) & ~255
buf = torch.empty(n * slot + 256, dtype=torch.uint8, device="cuda")
for k, s in enumerate(streams):
    buf[k * slot:k * slot + s.size].copy_(torch.from_numpy(s))
ref = np.asarray(Image.open(io.BytesIO(datas[0].tobytes())).convert("RGB"))[:, :, ::-1]
for _ in range(2):
    frames, status = ops.jpeg_decode_device(buf, slot, infos)
torch.cuda.synchronize()
best = 1e9
for _ in range(3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    frames, status = ops.jpeg_decode_device(buf, slot, infos)
    e1.record()
    torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1))
print(f"  {best:.2f} ms per 32 frames = {n / best * 1e3:.0f} frames/s, status {status.cpu().tolist()[:2]}, exact {bool(np.array_equal(frames[0].cpu().numpy(), ref))}", flush=True)
'''
for name in sys.argv[1:]:
    env = dict(os.environ)
    if name != "main":
        env["FACET_B200_LIB"] = os.path.abspath(f"facet_b200/variants/lib_{name}.so")
    print(name, flush=True)
    subprocess.run([sys.executable, "-c", CHILD], env=env)
