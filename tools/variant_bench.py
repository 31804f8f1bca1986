import sys, json, time
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import webp_decoder_b200 as W
from webp_decoder_b200 import parse as P
files=["noise_1920x1080_q75.webp","rgbgrad_1920x1080_q75.webp","checker_1920x1080_q75.webp","diag_1920x1080_q75.webp"]
pf=P.parse_batch([(ROOT / 'bench_data' / f).read_bytes() for f in files], pinned=True)
ctx=W.Context(0)
for name,sel in [("mix",[0,1,2,3]),("noise",[0]),("rgbgrad",[1]),("checker",[2]),("diag",[3])]:
    order=[sel[i%len(sel)] for i in range(1024)]
    kfs=[pf.kfs[i] for i in order]; frs=[pf.frames[i] for i in order]
    b=ctx.upload(kfs,frs)
    for kern in (3,2):
        ctx.set_kernel(kern)
        for mode in ("fused","recon_only","staged"):
            for it in range(3):
                if it==1: ctx.kernel_time()
                if mode=="fused": ctx.run(b,True,W.TIGHT)
                elif mode=="recon_only": ctx.run(b,False,W.TIGHT)
                else:
                    ctx.run(b,False,W.PADDED); ctx.filter(b)
            ms,n=ctx.kernel_time()
            print(f"{name:8s} kernel{kern} {mode:10s} {ms/2:.2f} ms per 1024 frames ({n} launches)")
    b.free()
