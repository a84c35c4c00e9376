#!/usr/bin/env python
"""Differential fuzzing of K2 / K3 (host SIMT emulator, tests/simt_emu): ses_rank_desc in both builds (fused / separate
kernels; float64 keys incl. +-inf, denormals, -0.0, constant vectors, NaNs of both signs; integer keys) against
np.flip(np.argsort(kind="stable")), and ses_update_openai / ses_materialize / ses_update_elite_mean with random layouts
against the C twin.  No GPU needed.

    python tools/emu_fuzz_k23.py <first_case> <n_cases>      (4 600 cases, 0 mismatches at the end of round 1)
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from simt_emu.emu_engine import EmuEngine
from oracle import twin
twin.build()
bad=0; t0=time.time()
for case in range(int(sys.argv[1]), int(sys.argv[1])+int(sys.argv[2])):
    rng=np.random.default_rng(case)
    os.environ["SES_K2_FUSED"]=str(case&1)
    n=int(rng.choice([2,3,31,32,33,255,256,257,1023,1024,1025, int(rng.integers(2,6000))]))
    kind=rng.choice(["float","ties","int","const","inf","nan"])
    E=int(rng.choice([1,5,7])); ms=int(rng.choice([500,37,1]))
    eng=EmuEngine(population=n, group=n, eval_ep_num=E, max_step=ms, seed=case)
    if kind=="float": r=rng.normal(0,100,n)
    elif kind=="ties": r=np.round(rng.normal(0,2,n)); r[rng.random(n)<0.2]=-0.0
    elif kind=="const": r=np.full(n, float(rng.integers(-3,3)))
    elif kind=="inf": r=rng.normal(0,1,n); r[rng.random(n)<0.1]=np.inf; r[rng.random(n)<0.1]=-np.inf; r[rng.random(n)<0.05]=1e-310
    elif kind=="nan":
        r=rng.normal(0,1,n); r[rng.random(n)<0.1]=np.inf; r[rng.random(n)<0.1]=-np.inf
        for b in (0x7ff8000000000000, 0xfff8000000000000, 0x7ff0000000000001, 0xfff0000000000123):
            r[rng.random(n)<0.05]=np.array([b],np.uint64).view(np.float64)[0]
    else: r=rng.integers(E, E*ms+1, n)/E
    want=np.flip(np.argsort(r,kind="stable")).astype(np.int32)
    ok=np.array_equal(eng.rank_desc(r, full_key=True), want)
    if kind=="int":
        o,sh=eng.rank_desc(r, shaped=True)
        ok = ok and np.array_equal(o,want) and np.array_equal(sh, twin.centered_rank(want))
    # K3 with this population: regenerated-noise gradient vs twin, random layout
    if n<=1500:
        group=int(rng.choice([n, max(1,n//4)])); n_head=int(rng.integers(0,min(2,group)+1)); n_par=(n-1)//group+1
        anti=bool(rng.random()<0.3); twin.set_antithetic(anti)
        e2=EmuEngine(population=n, group=group, n_head=n_head, n_parents=n_par, seed=case, antithetic=anti)
        shaped=twin.centered_rank(rng.permutation(n).astype(np.int32))
        mu=rng.normal(0,1,226).astype(np.float32); m=rng.normal(0,.01,226).astype(np.float32); v=np.abs(rng.normal(0,.01,226)).astype(np.float32)
        mu0,m0,v0=mu.copy(),m.copy(),v.copy()
        g=e2.update_openai(case, 0.3, 0.1, 3, shaped, mu, m, v)
        tg=twin.grad_openai(shaped,226,case,case,group,n_head,-(0.1/(n*0.3)))
        th,mm,vv=twin.adam(mu0,m0,v0,tg,e2.adam_a(0.1,3))
        ok = ok and np.array_equal(g,tg) and np.array_equal(mu,th) and np.array_equal(m,mm) and np.array_equal(v,vv)
        par=rng.normal(0,1,(n_par,226)).astype(np.float32)
        ids=rng.integers(0,n,min(n,40)).astype(np.int32)
        ok = ok and np.array_equal(e2.materialize(case,0.7,par,ids), twin.materialize(par,0.7,case,case,group,n_head,ids))
        k=int(rng.integers(1,min(n,20)+1)); order=rng.permutation(n).astype(np.int32)
        ok = ok and np.array_equal(e2.elite_mean(case,0.7,par,order,k), twin.elite_mean(twin.materialize(par,0.7,case,case,group,n_head,order[:k])))
        twin.set_antithetic(False)
    if not ok: bad+=1; print("MISMATCH", case, kind, n)
print("cases", sys.argv[2], "bad", bad, "time %.1f"%(time.time()-t0))
