import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
from test_training import _tiny, md
from neo360_b200 import training, synth
from oracle import neo360_oracle as orc
cuda=torch.device('cuda:0')
net, sc, P, rays, (W,H,nc,nf) = _tiny(cuda)
Pg={k:v.clone().requires_grad_(True) for k,v in P.items()}
maps={k:sc[k].clone().requires_grad_(True) for k in ("planes_xz","planes_xy","planes_yz","latent")}
osc=orc.Scene(maps["planes_xz"],maps["planes_xy"],maps["planes_yz"],maps["latent"],sc["src_poses"],float(sc["src_focal"][0]),float(sc["src_c"][0,0]),float(sc["src_c"][0,1]),W,H)
target=torch.rand(rays["rays_o"].shape[0],3,generator=torch.Generator().manual_seed(9))
mode=sys.argv[1] if len(sys.argv)>1 else "full"
def loss_fn(ret,tgt):
    if mode=="full": return training.training_loss(ret,tgt)
    if mode=="c0": return ((ret[0][0]-tgt)**2).mean()
    if mode=="c1": return ((ret[1][0]-tgt)**2).mean()
    if mode=="w": return (ret[1][1]**2).sum()+(ret[1][2]**2).sum()
ref=orc.render(rays,osc,Pg,nc,nf,white_bkgd=False,out_depth=False)
loss_fn(ref,target).backward()
dmaps={k:sc[k].to(cuda).requires_grad_(True) for k in maps}
batch={k:v.to(cuda) for k,v in rays.items()}; batch.update(dmaps); batch.update({k:sc[k].to(cuda) for k in ("src_poses","src_focal","src_c")})
batch["src_imgs"]=torch.zeros(3,3,H,W,device=cuda)
got=net(batch,False,False,None,None,out_depth=False)
loss_fn(got,target.to(cuda)).backward()
for name,p in net.named_parameters():
    g=Pg[name].grad
    if g is None: print(name,"ref None", None if p.grad is None else float(p.grad.abs().max())); continue
    if p.grad is None: print(name,"ours None", float(g.abs().max())); continue
    print(f"{name:45s} scale {float(g.abs().max()):.3e} err {md(p.grad,g):.3e}")
for k in maps: print(k, float(maps[k].grad.abs().max()), md(dmaps[k].grad,maps[k].grad))
