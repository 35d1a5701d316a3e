"""Where the 1e-5 bound on dark detector pixels comes from (CPU model, no GPU): the fused / tensor kernels carry the
phase in 2^-22 half-turn fixed point and take sin / cos from the SFU (absolute error 2^-21.4); both put an absolute
floor under every detector AMPLITUDE, so the relative error of a pixel grows as 1 / sqrt(pixel / brightest pixel).
Prints the relative error of the darkest 5x5 detector pixel at r0 = 0.08 m with FP64 accumulation for each source.

    python tools/dark_pixel_error_model.py --pupil 512 --r0 0.20 --obs-dim 2

also prints, per source, the largest amplitude error relative to the brightest pixel's amplitude (the floor f of
dP = 2 f sqrt(P P_max)), with a fourth source: the tensor cores truncate their FP32 accumulation, so the DM phase of the
4 main MMAs of a 64-deep K block loses up to one FP32 ulp of the running sum each, always towards zero.  That error has
the sign and the smoothness of the DM surface, so it adds up coherently over the pupil: it sets a floor of a few 1e-7
of the peak amplitude at any pupil size, where the random sources (quantisation, SFU) fall as 1 / sqrt(lit pixels)."""
import argparse
import numpy as np, sys
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adaptive_optics_gym_b200.tables import AOConfig, build_tables
from oracle.ao_oracle import hcipy_make_pupil_grid, hcipy_Cn_squared_from_fried_parameter, von_karman_screen
ap_=argparse.ArgumentParser()
ap_.add_argument('--pupil', type=int, default=240)
ap_.add_argument('--r0', type=float, default=0.08)
ap_.add_argument('--obs-dim', type=int, default=5)
args=ap_.parse_args()
N=args.pupil
cfg=AOConfig(fried_parameter=args.r0,num_modes=64,obs_dim=args.obs_dim,num_pupil_pixels=N)
T=build_tables(cfg,rng=np.random.default_rng(0))
g=hcipy_make_pupil_grid(N,0.5)
m1=T['mft_obs_1']; m2=T['mft_obs_2']; ap=T['aperture'].reshape(N,N)
lam=cfg.wavelength_wfs
rng=np.random.default_rng(5)
for s in range(4):
    scr=von_karman_screen(g,hcipy_Cn_squared_from_fried_parameter(args.r0,2.2e-6),10.0,np.random.default_rng(20+s)).reshape(N,N)
    a=rng.normal(0,1,64)/(np.arange(64)+10); surf=(T['dm_modes'].T@a).reshape(N,N); surf*=0.1*2.2e-6/surf.std()
    phi=scr/lam+2*surf*2*np.pi/lam
    def obs(ph, sc=None):
        E=ap*np.exp(1j*ph) if sc is None else ap*(sc[0]+1j*sc[1])
        F=m1@E@m2
        return np.abs(F)**2
    ref=obs(phi)
    # (1) phase quantisation 2^-22 half-turns (atmosphere tile) + DM rounding to same grid
    q=np.pi/2**22
    ph_q=np.round(scr/lam/q)*q+np.round(2*surf*2*np.pi/lam/q)*q
    e1=np.abs(obs(ph_q)-ref)/ref
    # (2) MUFU error model: abs error uniform +-2^-21.4 on sin and cos
    err=2**-21.4
    c=np.cos(phi)+rng.uniform(-err,err,phi.shape); sn=np.sin(phi)+rng.uniform(-err,err,phi.shape)
    e2=np.abs(obs(None,(c,sn))-ref)/ref
    # (3) fp32 rounding of sin, cos
    c=np.cos(phi).astype(np.float32).astype(float); sn=np.sin(phi).astype(np.float32).astype(float)
    P3=obs(None,(c,sn)); e3=np.abs(P3-ref)/ref
    # (4) truncating FP32 accumulation of the DM phase on the tensor cores (half-turns, 4 main MMAs per K block)
    d=2*surf*2/lam; ulp=np.spacing(np.abs(d).astype(np.float32)).astype(float)
    P4=obs(phi-np.pi*np.sign(d)*ulp*rng.uniform(0,1,(4,)+d.shape).sum(0))
    amp=lambda P: np.abs(np.sqrt(P)-np.sqrt(ref)).max()/np.sqrt(ref.max())
    floors=dict(zip(('phase-quant','mufu','fp32','tc-trunc'), (amp(obs(ph_q)), amp(obs(None,(np.cos(phi)+rng.uniform(-err,err,phi.shape),np.sin(phi)+rng.uniform(-err,err,phi.shape)))), amp(P3), amp(P4))))
    print(f'screen {s}: amplitude floor / peak amplitude: ' + '  '.join(f'{k} {v:.1e}' for k, v in floors.items()))
    print(f'screen {s}: min pixel / max {ref.min()/ref.max():.2e}; rel err max: phase-quant {e1.max():.2e}  mufu {e2.max():.2e}  fp32 {e3.max():.2e}')
