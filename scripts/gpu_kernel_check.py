"""Kernel-by-kernel numerical check on a B200 against torch fp32 (prints one line per case, never stops early).
Development aid; the pytest suite (tests/ -m gpu) is the gate."""
import os, sys, time, traceback
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F
import unet_pytorch_b200 as b2u
from unet_pytorch_b200 import ops

dev = torch.device("cuda:0")
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
RESULTS = []

def rel(a, b):
    a = a.float(); b = b.float()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()

def report(name, err, tol):
    ok = err <= tol
    RESULTS.append((name, err, tol, ok))
    print(f"{'PASS' if ok else 'FAIL'} {name}: err={err:.3e} tol={tol:.1e}", flush=True)

def run(name, fn):
    try:
        fn()
        torch.cuda.synchronize()
    except Exception as e:
        RESULTS.append((name, float('nan'), 0, False))
        print(f"FAIL {name}: EXC {type(e).__name__}: {e}", flush=True)
        traceback.print_exc()

def nhwc(x):  # NCHW fp32 -> NHWC bf16
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)

def nchw(x):  # NHWC bf16 -> NCHW fp32
    return x.float().permute(0, 3, 1, 2).contiguous()

def conv_case(N, H, W, C0, C1, Cout, taps, relu, bn=0):
    def f():
        g = torch.Generator(device="cpu").manual_seed(1)
        k = 3 if taps == 9 else 1
        x = torch.randn(N, C0 + C1, H, W, generator=g).to(dev)
        w = (torch.randn(Cout, C0 + C1, k, k, generator=g) / ((C0 + C1) * taps) ** 0.5).to(dev)
        b = torch.randn(Cout, generator=g).to(dev)
        xb = nhwc(x); xr = nchw(xb)
        wf, wd = ops.pack_weights(w)
        wr = w.to(torch.bfloat16).float()
        x0 = xb[..., :C0].contiguous(); x1 = xb[..., C0:].contiguous() if C1 else None
        y = ops.conv_fprop(x0, wf, b, Cout, taps=taps, relu=relu, x1=x1, bn=bn)
        ref = F.conv2d(xr, wr, b, padding=k // 2)
        if relu: ref = ref.relu()
        report(f"fprop N{N} {H}x{W} C{C0}+{C1}->{Cout} t{taps} bn{bn}", rel(nchw(y), ref), 6e-3)
        # dgrad
        dz = torch.randn(N, Cout, H, W, generator=g).to(dev)
        dzb = nhwc(dz); dzr = nchw(dzb)
        ref_dx = F.conv_transpose2d(dzr, wr, padding=k // 2)
        if C1:
            d0, d1 = ops.conv_dgrad(dzb, wd, C0, taps=taps, C1=C1)
            got = torch.cat([nchw(d0), nchw(d1)], 1)
            report(f"dgrad(split) same", rel(got, ref_dx), 6e-3)
        else:
            mask = nhwc(torch.randn(N, C0, H, W, generator=g).to(dev))
            d0 = ops.conv_dgrad(dzb, wd, C0, taps=taps, mask=mask)
            report(f"dgrad(mask) same", rel(nchw(d0), ref_dx * (nchw(mask) > 0)), 6e-3)
        # wgrad
        ref_dw = torch.nn.grad.conv2d_weight(xr, w.shape, dzr, padding=k // 2)
        dw = ops.conv_wgrad(x0, dzb, taps=taps, x1=x1)
        report(f"wgrad same", rel(dw, ref_dw), 2e-3)
        db = ops.bias_grad(dzb)
        report(f"bias_grad same", rel(db, dzr.sum((0, 2, 3))), 1e-4)
    run(f"conv N{N} {H}x{W} C{C0}+{C1}->{Cout} t{taps}", f)

def first_layer_case(N, H, W, Cout=64):
    def f():
        g = torch.Generator(device="cpu").manual_seed(2)
        x = torch.rand(N, 3, H, W, generator=g).to(dev)
        w = (torch.randn(Cout, 3, 3, 3, generator=g) / 27 ** 0.5).to(dev)
        b = torch.randn(Cout, generator=g).to(dev)
        col = ops.im2col_first(x)
        wf = ops.pack_weights_first(w)
        y = ops.conv_fprop(col, wf, b, Cout, taps=1, relu=True)
        ref = F.conv2d(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), b, padding=1).relu()
        report(f"first conv fprop N{N} {H}x{W}", rel(nchw(y), ref), 6e-3)
        dz = torch.randn(N, Cout, H, W, generator=g).to(dev)
        dzb = nhwc(dz)
        dw = ops.conv_wgrad(col, dzb, taps=1, first_cin=3)
        ref_dw = torch.nn.grad.conv2d_weight(x.to(torch.bfloat16).float(), w.shape, nchw(dzb), padding=1)
        report(f"first conv wgrad N{N} {H}x{W}", rel(dw, ref_dw), 2e-3)
    run("first layer", f)

def pool_up_case(N, H, W, C):
    def f():
        g = torch.Generator(device="cpu").manual_seed(3)
        x = torch.randn(N, C, H, W, generator=g).to(dev).relu()
        xb = nhwc(x); xr = nchw(xb).requires_grad_(True)
        y = ops.maxpool2x2(xb)
        ref = F.max_pool2d(xr, 2, 2)
        report(f"maxpool fwd {H}x{W} C{C}", rel(nchw(y), ref), 0.0)
        dp = nhwc(torch.randn(N, C, H // 2, W // 2, generator=g).to(dev))
        dsk = nhwc(torch.randn(N, C, H, W, generator=g).to(dev))
        ref.backward(nchw(dp))
        refdz = (xr.grad + nchw(dsk)) * (xr > 0)
        dz = ops.maxpool2x2_bwd(dp, xb, dskip=dsk, relu_mask=True)
        report(f"maxpool bwd {H}x{W} C{C}", rel(nchw(dz), refdz), 4e-3)
        # upsample
        xr2 = nchw(xb).requires_grad_(True)
        up = ops.upsample2x(xb)
        refu = F.interpolate(xr2, scale_factor=2, mode="bilinear", align_corners=True)
        report(f"upsample fwd {H}x{W} C{C}", rel(nchw(up), refu), 4e-3)
        du = nhwc(torch.randn(N, C, 2 * H, 2 * W, generator=g).to(dev))
        refu.backward(nchw(du))
        dl = ops.upsample2x_bwd(du, ylow=xb)
        report(f"upsample bwd {H}x{W} C{C}", rel(nchw(dl), xr2.grad * (xr2 > 0)), 4e-3)
    run(f"pool/up {H}x{W} C{C}", f)

def head_loss_case(N, H, W, C, onehot):
    def f():
        g = torch.Generator(device="cpu").manual_seed(4)
        x = torch.randn(N, 64, H, W, generator=g).to(dev).relu()
        xb = nhwc(x); xr = nchw(xb).requires_grad_(True)
        w = (torch.randn(C, 64, 1, 1, generator=g) / 8).to(dev).requires_grad_(True)
        b = torch.randn(C, generator=g).to(dev).requires_grad_(True)
        logits = ops.head_fwd(xb, w.detach().reshape(C, 64).contiguous(), b.detach())
        ref = F.conv2d(xr, w, b)
        report(f"head fwd C{C}", rel(logits, ref), 1e-5)
        png = torch.randint(0, C + 1, (N, H, W), generator=g).to(dev)
        oh = torch.eye(C + 1, device=dev)[png].contiguous()
        cw = (torch.rand(C, generator=g) + 0.5).to(dev)
        # reference losses (formulas of nets/unet_training.py restated with torch ops)
        lg = ref
        ce = F.cross_entropy(lg, png, weight=cw, ignore_index=C)
        lp = -F.cross_entropy(lg, png, weight=cw, ignore_index=C, reduction="none")
        focal = (-((1 - lp.exp()) ** 2) * (0.5 * lp)).mean()
        p = lg.permute(0, 2, 3, 1).reshape(N, -1, C).softmax(-1)
        t = oh.view(N, -1, C + 1)[..., :-1]
        tp = (t * p).sum((0, 1)); fp = p.sum((0, 1)) - tp; fn = t.sum((0, 1)) - tp
        dice = 1 - ((2 * tp + 1e-5) / (2 * tp + fn + fp + 1e-5)).mean()
        ph = (p > 0.5).float()
        tpf = (t * ph).sum((0, 1)); fpf = ph.sum((0, 1)) - tpf; fnf = t.sum((0, 1)) - tpf
        fs = ((2 * tpf + 1e-5) / (2 * tpf + fnf + fpf + 1e-5)).mean()
        out = ops.loss_fwd(logits, target=png, onehot=oh if onehot else None, cls_w=cw)
        report(f"CE C{C} oh{onehot}", abs(out[0].item() - ce.item()) / abs(ce.item()), 2e-5)
        report(f"Focal C{C}", abs(out[1].item() - focal.item()) / abs(focal.item()), 2e-5)
        report(f"Dice C{C}", abs(out[2].item() - dice.item()) / abs(dice.item()), 2e-5)
        report(f"fscore C{C}", abs(out[3].item() - fs.item()) / max(abs(fs.item()), 1e-9), 2e-5)
        for name, gs, loss in (("ce", [1, 0, 0], ce), ("focal", [0, 1, 0], focal), ("dice", [0, 0, 1], dice), ("ce+dice", [1, 0, 1], ce + dice)):
            gl, = torch.autograd.grad(loss, lg, retain_graph=True)
            dl = ops.loss_bwd(logits, out, torch.tensor(gs, dtype=torch.float32, device=dev), target=png, onehot=oh if onehot else None, cls_w=cw)
            report(f"dlogits {name} C{C}", rel(dl, gl), 2e-4)
        # head bwd
        gl, = torch.autograd.grad(ce + dice, lg, retain_graph=True)
        (ce + dice).backward()
        dx, dw, db = ops.head_bwd(gl.contiguous(), xb, w.detach().reshape(C, 64).contiguous())
        report(f"head dx C{C}", rel(nchw(dx), xr.grad * (xr > 0)), 4e-3)
        report(f"head dw C{C}", rel(dw, w.grad), 1e-4)
        report(f"head db C{C}", rel(db, b.grad), 1e-4)
        am = ops.argmax_u8(logits)
        report(f"argmax C{C}", (am.long() != logits.argmax(1)).float().mean().item(), 0.0)
    run(f"head/loss C{C}", f)

def hist_case(n, L, dtype=torch.uint8):
    def f():
        import numpy as np
        g = torch.Generator(device="cpu").manual_seed(5)
        a = torch.randint(0, n, (L,), generator=g).to(dtype)
        a[torch.rand(L, generator=g) < 0.03] = 255 if dtype == torch.uint8 else -1
        b = a.clone(); m = torch.rand(L, generator=g) < 0.2
        b[m] = torch.randint(0, n, (int(m.sum()),), generator=g).to(dtype)
        b[b >= n] = 0
        hist = torch.zeros(n * n + 1, dtype=torch.int64, device=dev)
        ops.fast_hist_accumulate(a.to(dev), b.to(dev), n, hist)
        an, bn_ = a.numpy().astype(np.int64), b.numpy().astype(np.int64)
        k = (an >= 0) & (an < n)
        ref = np.bincount(n * an[k] + bn_[k], minlength=n * n).reshape(n, n)
        got = hist[:-1].cpu().numpy().reshape(n, n)
        report(f"fast_hist n={n} L={L} {dtype}", float(np.abs(got - ref).sum()) + float(hist[-1].item()), 0.0)
    run(f"hist n={n}", f)

def adam_case():
    def f():
        g = torch.Generator(device="cpu").manual_seed(6)
        n = 4096 * 3
        p = torch.randn(n, generator=g).to(dev); p2 = p.clone().requires_grad_(True)
        opt = torch.optim.Adam([p2], lr=1e-3)
        m = torch.zeros_like(p); v = torch.zeros_like(p)
        for step in range(1, 4):
            gr = torch.randn(n, generator=g).to(dev)
            p2.grad = gr.clone(); opt.step()
            ops.adam_step(p, gr, m, v, step, 1e-3)
        report("adam 3 steps", rel(p, p2.detach()), 1e-6)
    run("adam", f)

if __name__ == "__main__":
    t0 = time.time()
    print("device:", torch.cuda.get_device_name(0), "SMs", b2u._lib.lib().b2u_num_sms(), flush=True)
    pool_up_case(2, 16, 32, 64)
    pool_up_case(1, 8, 8, 128)
    head_loss_case(2, 32, 48, 21, False)
    head_loss_case(2, 32, 48, 2, True)
    hist_case(21, 512 * 512 * 3 + 5)
    hist_case(2, 100003)
    hist_case(4, 70000, torch.int64)
    adam_case()
    first_layer_case(2, 32, 48)
    conv_case(1, 8, 16, 64, 0, 64, 9, True)        # single tile
    conv_case(2, 32, 48, 64, 0, 64, 9, True)
    conv_case(2, 24, 40, 128, 0, 128, 9, True)     # ragged tiles
    conv_case(1, 16, 16, 256, 0, 256, 9, False)
    conv_case(1, 16, 16, 512, 0, 512, 9, True)
    conv_case(1, 16, 32, 64, 128, 64, 9, True)     # virtual concat, dgrad N tile 192
    conv_case(1, 16, 16, 512, 512, 512, 9, True)
    conv_case(1, 4, 4, 512, 0, 512, 9, True)       # image smaller than the tile
    conv_case(2, 16, 16, 64, 0, 128, 1, False)     # 1x1
    conv_case(1, 64, 64, 128, 256, 128, 9, True)   # dgrad 384 = 2 x 192
    nfail = sum(1 for r in RESULTS if not r[3])
    print(f"SUMMARY: {len(RESULTS) - nfail} passed, {nfail} failed, {time.time() - t0:.1f}s")
