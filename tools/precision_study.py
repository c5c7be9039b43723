import os, sys, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import temporal_model_oracle as orc
torch.set_num_threads(8)
ARC=[3,3,3,3,3]; C=1024; N=256
sd=orc.make_state_dict(17,2,17,ARC,C,seed=0)
x=orc.make_input(N,243,seed=78)
def bf(t): return t.to(torch.bfloat16).float()
def split(t, planes):  # value represented
    if planes==2:
        hi=bf(t); return hi+bf(t-hi)
    return bf(t)
def run(cfg):
    # cfg: dict with per-layer operand precision 'x3' or 'bf', act planes for X (residual stream) and H
    eps=1e-5
    def aff(p):
        s=sd[p+'.weight']/torch.sqrt(sd[p+'.running_var']+eps); return s, sd[p+'.bias']-sd[p+'.running_mean']*s
    def gemm(a, w, prec):  # a [M,K] fp32 exact value; w [N,K]
        if prec=='x3': return a@w.T   # ~fp32
        if prec=='a2': return a@bf(w).T  # activations 2-plane exact, weights bf16
        return bf(a)@bf(w).T
    h=x.reshape(N,81,102)
    w0=sd['expand_conv.weight'].permute(0,2,1).reshape(C,102)
    s,b=aff('expand_bn')
    X=torch.relu(gemm(h.reshape(-1,102), w0, cfg['L'][0])*s+b)
    X=split(X,cfg['xp'])
    L=81
    for i in range(4):
        w1=sd[f'layers_conv.{2*i}.weight'].permute(0,2,1).reshape(C,3*C)
        w2=sd[f'layers_conv.{2*i+1}.weight'][:,:,0]
        M=X.shape[0]//3
        A=X.reshape(M,3*C)
        s,b=aff(f'layers_bn.{2*i}')
        Aop = A if cfg['L'][1+2*i]!='bf' else (bf(A) if cfg['xp']==2 else A)
        H=torch.relu(gemm(Aop,w1,cfg['L'][1+2*i])*s+b); H=split(H,cfg['hp'])
        s,b=aff(f'layers_bn.{2*i+1}')
        Z=torch.relu(gemm(H,w2,cfg['L'][2+2*i])*s+b)
        res=X.reshape(M,3,C)[:,1]
        X=split(res+Z,cfg['xp'])
    y=gemm(X, sd['shrink.weight'][:,:,0], cfg['L'][9])+sd['shrink.bias']
    return y.reshape(N,1,17,3)
ref=run(dict(L=['x3']*10,xp=2,hp=2))
# check ref vs oracle
yo=torch.from_numpy(orc.forward_numpy(sd,x[:4].numpy(),ARC)).float()
print('sim ref vs oracle', float((ref[:4]-yo).abs().max()/yo.abs().max()))
g=torch.Generator().manual_seed(5)
tgt=ref+torch.randn(ref.shape,generator=g)*0.03; tgt[:,:,0]=ref[:,:,0]
def report(name,cfg):
    y=run(cfg)
    d=float(orc.mpjpe(y,ref))*1000; sh=(float(orc.mpjpe(y,tgt))-float(orc.mpjpe(ref,tgt)))*1000
    print(f'{name:40s} mpjpe(new,ref)={d:.3f}mm shift={sh:+.4f}mm rel={float((y-ref).abs().max()/ref.abs().max()):.2e}')
report('all bf16, 1 plane', dict(L=['bf']*10,xp=1,hp=1))
report('all bf16, X 2 planes(res exact)', dict(L=['bf']*10,xp=2,hp=1))
report('expand+shrink x3', dict(L=['x3']+['bf']*8+['x3'],xp=1,hp=1))
report('expand,blk3,4,shrink x3', dict(L=['x3']+['bf']*4+['x3']*5,xp=1,hp=1))
report('expand,blk3,4,shrink x3 + X2', dict(L=['x3']+['bf']*4+['x3']*5,xp=2,hp=1))
report('expand,blk2,3,4,shrink x3 + X2', dict(L=['x3']+['bf']*2+['x3']*7,xp=2,hp=1))
report('only blk1 conv bf16', dict(L=['x3','bf']+['x3']*8,xp=2,hp=2))
