"""tcgen05 forward vs the quantisation-exact emulation; small + full size, with timing."""
import sys, time
sys.path[:0] = ['.', 'oracle', 'tests']
import torch
import mlp_emul as E
from nerfpp_b200 import ops

torch.manual_seed(0)
ws = [torch.randn(o, i) * (2.0 / i) ** 0.5 for o, i in ((64, 32), (16, 64), (64, 31), (64, 64), (3, 64))]
params = torch.cat([w.reshape(-1) for w in ws]).cuda()
packed = ops.mlp_small_pack(params)
for n in (1, 100, 128, 129, 1000, 5000):
    x = torch.cat([torch.randn(n, 32).half().float(), torch.randn(n, 16)], -1)
    out = ops.mlp_small_fwd(packed, x.cuda(), None, 1, None)
    torch.cuda.synchronize()
    e_out = E.forward_backward(ws, x, torch.zeros(n, 4))[0]
    err = float((out.cpu() - e_out).abs().max() / e_out.abs().max())
    print(f"n={n:6d} F32_CAT  max rel err vs emulation {err:.2e}")
rays, s = 700, 192
n = rays * s
enc = torch.randn(n, 32).half().cuda()
dirs = torch.nn.functional.normalize(torch.randn(rays, 3), dim=-1).cuda()
sh = ops.sh_encode(dirs, 4)
keep = (torch.rand(n) > 0.2).to(torch.uint8).cuda()
out = ops.mlp_small_fwd(packed, enc, sh, s, keep)
x = torch.cat([enc.float().cpu(), sh.cpu().repeat_interleave(s, 0)], -1)
e_out = E.forward_backward(ws, x, torch.zeros(n, 4), keep.cpu())[0]
print(f"n={n} ENC16 max rel err vs emulation {float((out.cpu() - e_out).abs().max() / e_out.abs().max()):.2e}")
# timing at the BASELINE sizes
for npts in (4096 * 64, 4096 * 192):
    enc = torch.randn(npts, 32, device="cuda").half()
    sh = ops.sh_encode(torch.nn.functional.normalize(torch.randn(4096, 3, device="cuda"), dim=-1), 4)
    outb = torch.empty(npts, 4, device="cuda")
    for _ in range(3):
        ops.mlp_small_fwd(packed, enc, sh, npts // 4096, None, out=outb)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        ops.mlp_small_fwd(packed, enc, sh, npts // 4096, None, out=outb)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    print(f"{npts} pts: {ms * 1e3:.1f} us  -> {npts * 18688 / ms / 1e9:.1f} TFLOP/s algorithmic")
