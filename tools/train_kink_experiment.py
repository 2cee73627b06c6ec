"""CPU experiment behind the gradient tolerances of tests/test_train_backward_gpu.py: the training step on the float64
stand-ins (oracle/train_ops.py), once exact and four times with the FORWARD GEMM outputs perturbed by 1e-6 of their maximum
(the size of the GPU forward's rounding, 2e-6 max-norm): a pre-ReLU activation within that distance of zero changes
sign, its ReLU mask flips, and the gradient w.r.t. the MLP hidden layer (g_hid) moves by 1e-2 .. 1e-1 of its maximum at
that element -- orders of magnitude above rounding -- which reaches the keypoint-encoder gradient as 3e-3 .. 7e-3.
Output committed as profiles/r02_train_kink.txt."""
import sys, json, os, numpy as np, torch
ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0,ROOT)
import tools.train_diag as Dg
from tests import emul_ops
from e2e_multi_view_matching_b200 import ops,_lib
for f in Dg.PATCHED: setattr(ops,f,getattr(emul_ops,f))
_lib.require_cuda=lambda d,w:None
name='mv3_64'
z=np.load(os.path.join(ROOT,'tests','golden','train_backward_%s.npz'%name)); case=json.loads(str(z['meta']))
data_np,sd=Dg.build(case)
f64,b64,r64,l64=Dg.run(case,sd,data_np,'cpu')
base_lin=emul_ops.linear
for seed in range(4):
    g=torch.Generator().manual_seed(seed)
    def noisy(a,w,bias=None,a2=None,residual=None,relu=False,alpha=1.0,tc_passes=0,presplit=False):
        y=base_lin(a,w,bias,a2,residual,relu,alpha)
        if tc_passes=='h16':   # forward GEMMs only: error like the GPU's (2e-6 of the max)
            y=y+torch.randn(y.shape,generator=g)*(1e-6*float(y.abs().max()))
        return y
    ops.linear=noisy
    fn,bn,rn,ln=Dg.run(case,sd,data_np,'cpu')
    L=len(case['layers'])
    print('seed',seed,' '.join('L%d:%.1e'%(L-1-j,Dg.rel(a['g_hid'],b['g_hid'])[0]) for j,(a,b) in enumerate(zip(bn['layers'],b64['layers']))),'g_kenc %.1e'%Dg.rel(bn['g_kenc'],b64['g_kenc'])[0])
