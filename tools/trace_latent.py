"""Per-phase trace of the persistent latent kernel (PCD_LT_TRACE): for the last reverse step, per phase: the span from the
first CTA entering it to the last CTA leaving its barrier, the longest / mean per-CTA work time and the mean barrier wait."""
import os, sys, collections
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
# enc1 + enc2 are the head phase, dec1 + output.0 + output.2 + update the tail phase
NAMES = ["head (enc1+enc2)", "enc3 G", "enc3 N", "enc4 G", "enc4 N", "gf0 G", "gf0 N", "gf3 G", "gf3 N",
         "dec4 G", "dec4 N", "dec3 G", "dec3 N", "dec2 G", "dec2 N", "tail (dec1+out0+out2+update)"]
import torch
import pcd_b200
from oracle import pointdiff_oracle as O
B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
sd = O.make_synthetic_latent_checkpoint(num_points=256)
m = pcd_b200.LatentDiffusion(pcd_b200.SimplePointNetVAE(256), is_voxel_based=False)
m.load_state_dict(sd, strict=False)
m = m.eval().cuda()
zT = torch.randn(B, 256, generator=torch.Generator().manual_seed(5)).cuda()
for _ in range(2):
    m.sample(B, num_steps=20, z_T=zT, return_latent=True)
path = os.path.join(ROOT, "gpurun_out", "lt_trace.txt")
os.environ["PCD_LT_TRACE"] = path
m.sample(B, num_steps=20, z_T=zT, return_latent=True)
torch.cuda.synchronize()
del os.environ["PCD_LT_TRACE"]
ph = collections.defaultdict(list)
for line in open(path):
    b, i, t0, t1, t2 = line.split()
    ph[int(i)].append((int(b), int(t0), int(t1), int(t2)))
tot = 0.0
for i in sorted(ph):
    r = ph[i]
    start = min(x[1] for x in r); end = max(x[3] for x in r)
    work = [x[2] - x[1] for x in r]
    busy = [w for w in work if w > 300]
    wait = [x[3] - x[2] for x in r]
    tot += (end - start) / 1e3
    print(f"{NAMES[i] if i < len(NAMES) else i:30s} span {(end-start)/1e3:7.2f} us  work max {max(work)/1e3:7.2f} mean(busy, n={len(busy):3d}) "
          f"{(sum(busy)/max(len(busy),1))/1e3:7.2f}  barrier wait min {min(wait)/1e3:6.2f} mean {sum(wait)/len(wait)/1e3:6.2f}")
print(f"sum of spans {tot:.1f} us")
