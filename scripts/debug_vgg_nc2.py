import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch, torch.nn.functional as F
import unet_pytorch_b200 as b2u
import warm_parity as WP
torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
dev = torch.device("cuda:0")
fam, C, med = sys.argv[1] if len(sys.argv) > 1 else "unet_vgg", 2, True
model, T = WP.build_reference(fam, C); model = model.to(dev)
WP.warm_up(model, T, C, 512, 4, 200, dev, medical=med)
sd = {k: v.detach().clone() for k, v in model.reference_state_dict().items()}
imgs, pngs = WP.make_batch(8, C, 512, 7, med, dev)
z64, g64, l64 = WP.run_reference(model, T, imgs, pngs, C, torch.float64)
za, ga, la = WP.run_reference(model, T, imgs, pngs, C, torch.float32, autocast=True)
zo, go, lo = WP.run_product(b2u, fam, sd, imgs, pngs, C)
print("loss fp64", l64, "autocast", la, "ours", lo)
w = torch.ones(C, device=dev)
def ref_loss(z):
    z = z.double().clone().requires_grad_(True)
    l = WP.loss_of(T, z, pngs, C, w.double()); l.backward(); return l.item(), z.grad
def our_loss(z):
    z = z.float().clone().requires_grad_(True)
    labels = F.one_hot(pngs, C + 1).float()
    l = b2u.CE_Loss(z, pngs, w, num_classes=C) + b2u.Dice_loss(z, labels); l.backward(); return l.item(), z.grad
for name, z in (("z64", z64), ("ours", zo), ("autocast", za)):
    lr, gr = ref_loss(z); lo_, go_ = our_loss(z)
    print(f"logits={name}: ref-loss {lr:.6f} our-loss {lo_:.6f}  dlogits rel {((go_.double()-gr).norm()/gr.norm()).item():.2e}")
d = (zo.double() - z64)
print("logit diff mean per class", d.mean((0, 2, 3)).tolist(), "rms", d.pow(2).mean().sqrt().item(), "logit rms", z64.pow(2).mean().sqrt().item())
m64 = (z64[:, 1] - z64[:, 0]); mo = (zo[:, 1] - zo[:, 0]).double(); ma = (za[:, 1] - za[:, 0]).double()
print("margin diff ours: mean", (mo - m64).mean().item(), "rms", (mo - m64).pow(2).mean().sqrt().item(), " autocast: mean", (ma - m64).mean().item(), "rms", (ma - m64).pow(2).mean().sqrt().item())
sgn = torch.where(pngs == 1, 1.0, -1.0).double()
print("signed margin change (toward correct): ours", ((mo - m64) * sgn).mean().item(), "autocast", ((ma - m64) * sgn).mean().item())
# error of dlogits-from-reference-loss on each logits vs on z64
_, g0 = ref_loss(z64); _, g1 = ref_loss(zo); _, g2 = ref_loss(za)
print("dlogits(ref loss) ours-vs-64", ((g1 - g0).norm() / g0.norm()).item(), "autocast-vs-64", ((g2 - g0).norm() / g0.norm()).item())
for k in list(g64)[:4] + list(g64)[-4:]:
    print(k, WP._rel(go[k], g64[k]), WP._rel(ga[k], g64[k]))
