"""CLIP preprocess and pHash on 24 MP frames (32 per launch, CUDA events, best of 3 x 3)."""
import sys
import torch
sys.path.insert(0, ".")
sys.path.insert(0, "scripts")
from facet_b200 import ops
from time_tech import make_frames

n = 32
fr = make_frames("photo", n)
luma = torch.empty(fr.shape[:3], dtype=torch.uint8, device="cuda")
ops.tech_stats_raw(fr, luma_out=luma)


def best_ms(fn):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e9
    for _ in range(3):
        e0.record()
        for _ in range(3):
            fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / 3)
    return best


a = best_ms(lambda: ops.clip_preprocess(fr))
b = best_ms(lambda: ops.phash(fr, device_only=True, luma=luma))
print(f"clip_preprocess {a * 1e3 / n:.2f} us / frame, phash (luma ready) {b * 1e3 / n:.2f} us / frame")
