#!/usr/bin/env python
"""Randomised CPU parity sweep (no GPU): for every seed in [lo, hi) a regime-randomised fleet (synth MIX, 17..1100 instances),
every decision routine of the product (decide_stream with full and tiny windows/budgets, decide_fast 32/16, budgeted
single-lane decide_ctx) against the oracle on 600 mixed decisions each, and the instance-shard min-loc protocol (2/3/5/8
shards) against the unsharded result.  usage: random_sweep.py LO HI"""
import os, sys, ctypes as C, numpy as np, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from modelmesh_b200 import _lib
from modelmesh_b200.fleet import Fleet
from modelmesh_b200.sharding import combine_shard_keys, decode_shard_keys
from modelmesh_b200.synth import make_decisions, make_fleet, load_into_fleet
from helpers import oracle_from_synth, solver_from_synth, compare_decisions
from oracle import binding
binding.build()
lib = _lib.load(os.path.join(ROOT, "tests", "emul", "_build", "libmmplace_emul.so"), require_all=False)
lib.mmp_emul_set_keys.argtypes = [C.c_void_p, C.c_void_p]
lib.mmp_emul_lane_bails.restype = C.c_long
t0 = time.time(); bad = 0; n_dec = 0
lo, hi = int(sys.argv[1]), int(sys.argv[2])
for seed in range(lo, hi):
    ni = [17, 33, 64, 97, 160, 300, 520, 700, 1100][seed % 9]
    fl = make_fleet("MIX", 300, ni, seed)
    o = oracle_from_synth(fl)
    s = solver_from_synth(fl, lib)
    for shape, win, budget in ((2, 14, 64), (2, [1, 2, 3, 5][seed % 4], [2, 5, 64][seed % 3]), (32, 14, 64), (16, 14, 64), (1, 14, [3, 48][seed % 2])):
        lib.mmp_emul_set_window(shape); lib.mmp_emul_set_lane_window(win); lib.mmp_emul_set_lane_budget(budget)
        sd = make_decisions(fl, 600, seed * 7 + shape)
        try:
            compare_decisions(fl, sd, o, s, seed=seed + 5, full_lists=False)
        except AssertionError as e:
            bad += 1; print("MISMATCH seed", seed, "shape", shape, win, budget, str(e)[:300]); 
        n_dec += 600
    # sharded protocol
    world = [2, 3, 5, 8][seed % 4]
    lib.mmp_emul_set_window(2); lib.mmp_emul_set_lane_window(14); lib.mmp_emul_set_lane_budget(64)
    sd = make_decisions(fl, 600, seed)
    kw = dict(fresh=sd.fresh if len(sd.fresh) else None, extra=sd.extra if len(sd.extra) else None)
    ref = s.place_batch(sd.dec, fl.now_ms, 77, **kw)
    keys = []
    for r in range(world):
        f = Fleet(fl.min_space_units, fl.min_churn_age_ms, fl.default_model_size_units, fl.n_instances, fl.n_models, shard_rank=r, shard_count=world, lib=lib)
        load_into_fleet(fl, f)
        k = np.zeros(600, dtype=np.uint64); lib.mmp_emul_set_keys(f.h, k.ctypes.data_as(C.c_void_p))
        f.place_batch(sd.dec, fl.now_ms, 77, **kw); lib.mmp_emul_set_keys(f.h, None); f.close(); keys.append(k)
    t, c, op = decode_shard_keys(combine_shard_keys(np.stack(keys)))
    cl = ~op
    if not (np.array_equal(t[cl], ref["target"][cl]) and np.array_equal(c[cl], ref["n_candidates"][cl])):
        bad += 1; print("SHARD MISMATCH seed", seed, world)
    s.close()
print("seeds", lo, hi, "decisions", n_dec, "bad", bad, "sec %.0f" % (time.time() - t0))
