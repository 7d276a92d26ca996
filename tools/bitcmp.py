import argparse, os, sys, subprocess, torch
sys.path.insert(0, os.getcwd())
# run the same forward under two libraries (separate processes), compare bitwise
# --case picks the constructor: the default pro model (nearest+conv x4) never reaches the pixel-shuffle heads or the 3conv residual
CASES = {
    "pro": {},
    "3conv": dict(resi_connection="3conv"),
    "pixelshuffle2": dict(upsampler="pixelshuffle", upscale=2),
    "pixelshuffle3": dict(upsampler="pixelshuffle", upscale=3),
    "pixelshuffledirect4": dict(upsampler="pixelshuffledirect", upscale=4),
    "none": dict(upsampler=None, upscale=1),
}
ap = argparse.ArgumentParser()
ap.add_argument("--case", choices=sorted(CASES), default="pro")
ap.add_argument("libs", nargs=2)
args = ap.parse_args()
code = '''
import os, sys, torch
sys.path.insert(0, os.getcwd())
import hitsir_b200
torch.manual_seed(0)
m = hitsir_b200.HiT_SIR(True, True, True, **dict(hitsir_b200.PRO_KWARGS, **eval(sys.argv[2]))).eval()
sd = m.state_dict()
g = torch.Generator().manual_seed(1)
for k, v in sd.items():
    if v.dim() >= 2: sd[k] = torch.randn(v.shape, generator=g) * (0.4 / max(1, v[0].numel()) ** 0.5)
    else: sd[k] = torch.randn(v.shape, generator=g) * 0.1 + (1.0 if "norm" in k and k.endswith("weight") else 0.0)
m.load_state_dict(sd)
m = m.to("cuda:0")
x = torch.rand(2, 3, 100, 72, generator=g).to("cuda:0")
with torch.no_grad(): y = m(x)
torch.save(y.cpu(), sys.argv[1])
'''
outs = []
for lib in args.libs:
    env = dict(os.environ, HITSIR_B200_LIB=os.path.abspath(lib))
    out = f"/tmp/y_{args.case}_{os.path.basename(lib)}.pt"
    subprocess.run([sys.executable, "-c", code, out, repr(CASES[args.case])], env=env, check=True)
    outs.append(torch.load(out))
print(args.case, "shape", tuple(outs[0].shape), "bit-identical:", torch.equal(outs[0], outs[1]), "max diff", (outs[0] - outs[1]).abs().max().item(),
      "finite", torch.isfinite(outs[0]).all().item(), "absmax", outs[0].abs().max().item())
