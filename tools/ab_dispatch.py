"""Bit-for-bit A/B of two builds of libmbpo_b200.so on the host-dispatched entry points.

Runs every entry point whose host-side dispatch (System table, PRNG / math mode, policy checks) lives in the C
library on seeded inputs, and saves all outputs.  Run it twice, in two processes, against the two builds:

    MBPO_B200_LIB=/path/to/old/libmbpo_b200.so python tools/ab_dispatch.py save OUT/a.npz
    python tools/ab_dispatch.py compare OUT/a.npz OUT/ab_dispatch_report.json

`compare` runs the in-tree build, compares every array with the saved one bit for bit and writes a JSON report;
it exits non-zero on any difference.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                "model-based-policy-optimizers_b200"))
from mbpo_b200 import _lib as L  # noqa: E402

DEV = torch.device("cuda", 0)
PEND = L.PendulumParamsC(8.0, 2.0, 0.05, 10.0, 1.0, 1.0, 0.001, 1.0, 0.0)
GEN = L.GeneralSystemParamsC(PEND, 0.1, L.PointMassParamsC(0.1, 1.0, 2.0, 0.5, -0.5, 0.1, 0.01))
SYSTEMS = {"pendulum": (L.SYSTEM_PENDULUM, 3, 1), "noisy_pendulum": (L.SYSTEM_NOISY_PENDULUM, 3, 1),
           "point_mass": (L.SYSTEM_POINT_MASS, 4, 2)}


def _t(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a)).to(DEV, dtype)


def _keys(rng, n):
    return torch.from_numpy(rng.integers(0, 2**32, (n, 2), dtype=np.uint32)).to(DEV)


def _state(rng, E, X):
    if X == 3:
        th = rng.uniform(-np.pi, np.pi, E)
        return np.stack([np.cos(th), np.sin(th), rng.uniform(-8, 8, E)], -1).astype(np.float32)
    return rng.uniform(-1, 1, (E, X)).astype(np.float32)


def _policy(rng, X, A, num_hidden, kernel, keep):
    p = L.PolicyParamsC()
    p.num_hidden, p.hidden, p.obs_dim, p.action_dim = num_hidden, 64, X, A
    dims = [X] + [64] * num_hidden + [2 * A]
    for l in range(num_hidden + 1):
        w = _t(rng.normal(0, 1 / np.sqrt(dims[l]), (dims[l], dims[l + 1])))
        b = _t(rng.normal(0, 0.1, dims[l + 1]))
        keep += [w, b]
        p.w[l], p.b[l] = L.ptr(w), L.ptr(b)
    p.min_std, p.head, p.kernel = 0.001, L.HEAD_NORMAL_TANH, kernel
    for i in range(4):
        p.obs_mean[i], p.obs_std[i] = 0.0, 1.0
    return p


def run() -> dict:
    out = {}
    st = L.stream_ptr(DEV)
    rng = np.random.default_rng(1234)
    keep = []

    def chk(name, rc):
        if rc != L.MBPO_OK:
            raise RuntimeError("%s: %d %s" % (name, rc, L.lib.mbpo_last_error()))

    # PRNG primitives, replay randint
    keys = _keys(rng, 64)
    for mode in (0, 1):
        ks = torch.empty((64, 5, 2), dtype=torch.uint32, device=DEV)
        chk("split", L.lib.mbpo_prng_split(L.ptr(keys), 64, 5, mode, L.ptr(ks), st))
        bits = torch.empty((64, 7), dtype=torch.uint32, device=DEV)
        chk("bits", L.lib.mbpo_prng_random_bits(L.ptr(keys), 64, 7, mode, L.ptr(bits), st))
        uni = torch.empty((64, 7), device=DEV)
        chk("uniform", L.lib.mbpo_prng_uniform(L.ptr(keys), 64, 7, mode, -2.0, 3.0, L.ptr(uni), st))
        nrm = torch.empty((64, 7), device=DEV)
        chk("normal", L.lib.mbpo_prng_normal(L.ptr(keys), 64, 7, mode, L.ptr(nrm), st))
        ri = torch.empty((64, 7), dtype=torch.int32, device=DEV)
        chk("randint", L.lib.mbpo_prng_randint(L.ptr(keys), 64, 7, mode, -3, 1000, L.ptr(ri), st))
        out.update({"prng%d_split" % mode: ks, "prng%d_bits" % mode: bits, "prng%d_uniform" % mode: uni,
                    "prng%d_normal" % mode: nrm, "prng%d_randint" % mode: ri})

    # replay sample
    cap, width, n = 1000, 13, 700
    data = _t(rng.normal(size=(cap, width)))
    rs = L.ReplayStateC(data=L.ptr(data), capacity=cap, row_width=width, head=0, insert_position=n, sample_position=0)
    for mode in (0, 1):
        kout = torch.empty(2, dtype=torch.uint32, device=DEV)
        idx = torch.empty(256, dtype=torch.int32, device=DEV)
        batch = torch.empty((256, width), device=DEV)
        chk("replay_sample", L.lib.mbpo_replay_sample(C.byref(rs), L.ptr(keys[0]), mode, 256, L.ptr(kout), L.ptr(idx),
                                                      L.ptr(batch), st))
        out.update({"replay%d_key" % mode: kout, "replay%d_idx" % mode: idx, "replay%d_batch" % mode: batch})

    E, T, ep_len = 1000, 37, 11
    for sname, (kind, X, A) in SYSTEMS.items():
        x0 = _t(_state(rng, E, X))
        first = _t(_state(rng, E, X))
        steps0 = _t((rng.integers(0, ep_len, E)).astype(np.float32))
        done0 = _t((rng.uniform(size=E) < 0.2).astype(np.float32))
        sk = _keys(rng, E)
        acts = _t(rng.uniform(-1.2, 1.2, (T, E, A)))
        # System.step and the objective
        for mode in (0, 1):
            u = _t(rng.uniform(-1.5, 1.5, (E, A)))
            xn, r, ko = torch.empty_like(x0), torch.empty(E, device=DEV), torch.zeros_like(sk)   # ko: keyed only
            chk("step_general", L.lib.mbpo_system_step_general(kind, C.byref(GEN), mode, L.ptr(x0), L.ptr(u), L.ptr(sk),
                                                              E, L.ptr(xn), L.ptr(r), L.ptr(ko), st))
            out.update({"%s_step%d_x" % (sname, mode): xn, "%s_step%d_r" % (sname, mode): r,
                        "%s_step%d_k" % (sname, mode): ko})
            H, B, M = 15, 8, 64
            xo = x0[:B].contiguous()
            aa = _t(rng.uniform(-1, 1, (B, M, H, A)))
            kk = _keys(rng, B * M)
            for P, summ in ((0, 0), (3, 0), (3, 1)):
                v = torch.empty((B, M), device=DEV)
                ob = torch.empty((B, M, H, X), device=DEV) if P == 0 else None
                rw = torch.empty((B, M, H), device=DEV) if P == 0 else None
                chk("objective", L.lib.mbpo_system_objective(kind, C.byref(GEN), mode, H, L.ptr(xo), L.ptr(aa), L.ptr(kk),
                                                             B, M, P, summ, L.ptr(v), L.ptr(ob), L.ptr(rw), None, st))
                out["%s_obj%d_P%d_s%d" % (sname, mode, P, summ)] = v
                if P == 0:
                    out["%s_obj%d_obs" % (sname, mode)], out["%s_obj%d_rew" % (sname, mode)] = ob, rw
        # env unroll / rollout with every combination of NULL outputs
        combos = [(o, rest) for o in (True, False) for rest in ((1, 1, 1, 1), (1, 0, 1, 0), (0, 1, 0, 1), (1, 1, 0, 1))]
        modes = (0, 1)
        for mode in modes:
            for ci, (with_obs, rest) in enumerate(combos):
                for unroll in ((True, False) if kind == L.SYSTEM_PENDULUM else (True,)):
                    oo, so, do, ko = torch.empty_like(x0), torch.empty_like(steps0), torch.empty_like(done0), \
                        torch.empty_like(sk)
                    ob = torch.zeros((T, E, X), device=DEV) if with_obs else None
                    rw = torch.zeros((T, E), device=DEV) if rest[0] else None
                    dc = torch.zeros((T, E), device=DEV) if rest[1] else None
                    nx = torch.zeros((T, E, X), device=DEV) if rest[2] else None
                    tc = torch.zeros((T, E), device=DEV) if rest[3] else None
                    if kind == L.SYSTEM_PENDULUM and unroll:
                        chk("env_unroll", L.lib.mbpo_env_unroll(
                            kind, C.addressof(PEND), mode, 3, 1, ep_len, 1 + ci % 2, L.ptr(x0), L.ptr(steps0),
                            L.ptr(done0), L.ptr(oo), L.ptr(so), L.ptr(do), L.ptr(first), L.ptr(acts), E, T, L.ptr(ob),
                            L.ptr(rw), L.ptr(dc), L.ptr(nx), L.ptr(tc), st))
                    elif kind == L.SYSTEM_PENDULUM:
                        oo.copy_(x0); so.copy_(steps0); do.copy_(done0)
                        chk("env_rollout", L.lib.mbpo_env_rollout(
                            kind, C.addressof(PEND), mode, 3, 1, ep_len, 1, L.ptr(oo), L.ptr(so), L.ptr(do),
                            L.ptr(first), L.ptr(acts), E, T, L.ptr(ob), L.ptr(rw), L.ptr(dc), L.ptr(nx), L.ptr(tc),
                            st))
                    else:
                        chk("env_unroll_general", L.lib.mbpo_env_unroll_general(
                            kind, C.byref(GEN), mode, ep_len, 1 + ci % 2, L.ptr(x0), L.ptr(steps0), L.ptr(done0),
                            L.ptr(sk), L.ptr(oo), L.ptr(so), L.ptr(do), L.ptr(ko), L.ptr(first), L.ptr(acts), E, T,
                            L.ptr(ob), L.ptr(rw), L.ptr(dc), L.ptr(nx), L.ptr(tc), st))
                    tag = "%s_env%d_c%d_%s" % (sname, mode, ci, "unroll" if unroll else "rollout")
                    for fname, f in (("obs", oo), ("steps", so), ("done", do), ("key", ko), ("observation", ob),
                                     ("reward", rw), ("discount", dc), ("next_obs", nx), ("trunc", tc)):
                        if f is not None and (fname != "key" or kind == L.SYSTEM_NOISY_PENDULUM):
                            out[tag + "_" + fname] = f
        # the policy in the loop
        kernels = (L.ACTOR_CUDA_CORES, L.ACTOR_TCGEN05, L.ACTOR_TCGEN05_WIDE) if kind == L.SYSTEM_PENDULUM else \
            (L.ACTOR_CUDA_CORES,)
        for kernel in kernels:
            pol = _policy(rng, X, A, 3, kernel, keep)
            for prng in (0, 1):
                for math in ((0, 1) if kind == L.SYSTEM_PENDULUM else (0,)):
                    for conv in (L.KEYS_SAC, L.KEYS_UNROLL):
                        tag = "%s_actor_k%d_p%d_m%d_c%d" % (sname, kernel, prng, math, conv)
                        obs, stp, dn, sko = x0.clone(), steps0.clone(), done0.clone(), torch.empty_like(sk)
                        key = keys[prng].contiguous()
                        ao, ro, dco, no, to = (torch.empty((T, E, A), device=DEV), torch.empty((T, E), device=DEV),
                                               torch.empty((T, E), device=DEV), torch.empty((T, E, X), device=DEV),
                                               torch.empty((T, E), device=DEV))
                        kout = torch.empty(2, dtype=torch.uint32, device=DEV)
                        raw, lp = torch.empty((T, E, A), device=DEV), torch.empty((T, E), device=DEV)
                        if kind == L.SYSTEM_PENDULUM:
                            chk(tag, L.lib.mbpo_actor_rollout_extras(
                                kind, C.addressof(PEND), math, prng, C.byref(pol), 0, conv, L.ptr(key), ep_len, 1,
                                L.ptr(obs), L.ptr(stp), L.ptr(dn), L.ptr(first), E, T, L.ptr(ao), L.ptr(ro),
                                L.ptr(dco), L.ptr(no), L.ptr(to), L.ptr(kout), L.ptr(raw), L.ptr(lp), st))
                        else:
                            chk(tag, L.lib.mbpo_actor_rollout_general(
                                kind, C.byref(GEN), prng, C.byref(pol), 0, conv, L.ptr(key), ep_len, 1, L.ptr(obs),
                                L.ptr(stp), L.ptr(dn), L.ptr(sk), L.ptr(sko), L.ptr(first), E, T, L.ptr(ao),
                                L.ptr(ro), L.ptr(dco), L.ptr(no), L.ptr(to), L.ptr(kout), L.ptr(raw), L.ptr(lp), st))
                        for fname, f in (("obs", obs), ("steps", stp), ("done", dn), ("action", ao), ("reward", ro),
                                         ("discount", dco), ("next_obs", no), ("trunc", to), ("key", kout),
                                         ("raw", raw), ("log_prob", lp)):
                            out[tag + "_" + fname] = f
                        if kind == L.SYSTEM_NOISY_PENDULUM:
                            out[tag + "_sys_key"] = sko
        # the pendulum's reverse scan, time-major [T, E, ...] and dense [E, T, ...], with NULL cotangents
        if kind == L.SYSTEM_PENDULUM:
            obs_t = _t(_state(rng, E * T, X).reshape(T, E, X))
            cot = [_t(rng.normal(size=s)) for s in ((T, E), (T, E, X), (T, E, X), (T, E))]
            for layout in ("time_major", "dense"):
                f = (lambda v: v) if layout == "time_major" else (lambda v: v.transpose(0, 1).contiguous())
                ob, ac = f(obs_t), f(acts[..., 0])
                st_t, st_e = (E, 1) if layout == "time_major" else (1, T)
                sx_t, sx_e = (E * X, X) if layout == "time_major" else (X, T * X)
                for use in ((1, 1, 1, 1), (1, 0, 0, 0), (0, 1, 0, 1)):
                    gr, gn, go, ga = (f(c) if u else None for c, u in zip(cot, use))
                    g_act, g_x0 = torch.empty_like(ac), torch.empty((E, X), device=DEV)
                    chk("rollout_adjoint", L.lib.mbpo_rollout_adjoint(
                        kind, C.addressof(PEND), X, A, E, T, st_t, st_e, sx_t, sx_e, L.ptr(ob), L.ptr(ac), L.ptr(gr),
                        L.ptr(gn), L.ptr(go), L.ptr(ga), L.ptr(g_act), L.ptr(g_x0), st))
                    tag = "%s_adjoint_%s_%d%d%d%d" % ((sname, layout) + use)
                    out.update({tag + "_g_action": g_act, tag + "_g_x0": g_x0})
        # the plans, fused and staged
        params = C.addressof(PEND) if kind == L.SYSTEM_PENDULUM else C.addressof(GEN)
        for prng in (0, 1):
            for math in ((0, 1) if kind == L.SYSTEM_PENDULUM else (0,)):
                cfg = L.IcemCfgC()
                chk("cfg", L.lib.mbpo_icem_cfg_init(C.byref(cfg), 20, A, X, 3, 128, 16, 0.5, 0.1, 3, 0.0, 0.3, -1.0,
                                                    1.0, 1, 1e4))
                cfg.prng_mode, cfg.system_kind, cfg.math_mode = prng, kind, math
                B = 6
                xo = x0[:B].contiguous()
                kin = keys[:B].contiguous()
                seq_in = _t(rng.uniform(-1, 1, (B, 20, A)))
                for fused in (True, False):
                    seq, val = torch.empty_like(seq_in), torch.empty(B, device=DEV)
                    kout = torch.empty((B, 2), dtype=torch.uint32, device=DEV)
                    if fused:
                        assert L.lib.mbpo_icem_plan_is_fused(C.byref(cfg)) == 1
                        chk("plan", L.lib.mbpo_icem_plan(C.byref(cfg), params, L.ptr(xo), L.ptr(kin),
                                                         L.ptr(seq_in), B, L.ptr(seq), L.ptr(val), L.ptr(kout), None,
                                                         st))
                    else:
                        nb = L.lib.mbpo_icem_workspace_bytes(C.byref(cfg), B)
                        ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
                        chk("plan_staged", L.lib.mbpo_icem_plan_staged(C.byref(cfg), params, L.ptr(xo),
                                                                       L.ptr(kin), L.ptr(seq_in), B, L.ptr(seq),
                                                                       L.ptr(val), L.ptr(kout), L.ptr(ws), nb, st))
                    tag = "%s_plan%d%d_%s" % (sname, prng, math, "fused" if fused else "staged")
                    out.update({tag + "_seq": seq, tag + "_val": val, tag + "_key": kout})
                if kind != L.SYSTEM_PENDULUM:
                    continue
                # the pendulum's fused plan at the flagship size (H = 30, 512 samples; white and colored noise), an
                # any-horizon instance (H = 23), cluster plans and the one-launch closed loop
                for H, exponent, B, cluster in ((30, 0.0, 40, 1), (30, 2.0, 40, 1), (30, 0.0, 1, 16), (30, 2.0, 3, 4),
                                                (23, 1.0, 5, 1)):
                    cfg = L.IcemCfgC()
                    chk("cfg", L.lib.mbpo_icem_cfg_init(C.byref(cfg), H, A, X, 1, 512, 50, 0.5, 0.1, 5, exponent,
                                                        0.3, -2.0, 2.0, 1, 1e4))
                    cfg.prng_mode, cfg.system_kind, cfg.math_mode = prng, kind, math
                    xo = _t(_state(rng, B, X))
                    kin = _keys(rng, B)
                    seq_in = _t(rng.uniform(-1, 1, (B, H, A)))
                    seq, val = torch.empty_like(seq_in), torch.empty(B, device=DEV)
                    kout = torch.empty((B, 2), dtype=torch.uint32, device=DEV)
                    chk("plan_clustered", L.lib.mbpo_icem_plan_clustered(
                        C.byref(cfg), params, L.ptr(xo), L.ptr(kin), L.ptr(seq_in), B, L.ptr(seq), L.ptr(val),
                        L.ptr(kout), None, cluster, st))
                    tag = "%s_plan%d%d_H%d_e%g_B%d_c%d" % (sname, prng, math, H, exponent, B, cluster)
                    out.update({tag + "_seq": seq, tag + "_val": val, tag + "_key": kout})
                    if H != 30 or exponent != 0.0:
                        continue
                    n_mpc = 4   # closed-loop steps (T above stays the env / actor rollout length)
                    sto, rwo = torch.empty((n_mpc, B, X), device=DEV), torch.empty((n_mpc, B), device=DEV)
                    aco, seq = torch.empty((n_mpc, B, A), device=DEV), torch.empty_like(seq_in)
                    kout = torch.empty((B, 2), dtype=torch.uint32, device=DEV)
                    chk("mpc", L.lib.mbpo_icem_mpc_closed_loop_clustered(
                        C.byref(cfg), params, L.ptr(xo), L.ptr(kin), L.ptr(seq_in), B, n_mpc, L.ptr(sto), L.ptr(rwo),
                        L.ptr(aco), L.ptr(seq), L.ptr(kout), cluster, st))
                    tag = "%s_mpc%d%d_H%d_B%d_c%d" % (sname, prng, math, H, B, cluster)
                    out.update({tag + "_states": sto, tag + "_rewards": rwo, tag + "_actions": aco, tag + "_seq": seq,
                                tag + "_key": kout})
    torch.cuda.synchronize(DEV)
    return {k: (v.cpu().view(torch.int32) if v.dtype == torch.uint32 else v.cpu()).numpy() for k, v in out.items()}


def main() -> int:
    torch.cuda.set_device(DEV)
    arrays = run()
    if sys.argv[1] == "save":
        np.savez(sys.argv[2], **arrays)
        print("saved %d arrays from %s" % (len(arrays), L.LIB_PATH))
        return 0
    ref = np.load(sys.argv[2])
    diff = sorted(k for k in arrays if k not in ref or arrays[k].tobytes() != ref[k].tobytes())
    missing = sorted(k for k in ref.files if k not in arrays)
    report = {"device": torch.cuda.get_device_name(DEV), "arrays": len(arrays),
              "values": int(sum(a.size for a in arrays.values())), "different": diff, "missing": missing}
    with open(sys.argv[3], "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps({k: v for k, v in report.items()}))
    return 1 if diff or missing else 0


if __name__ == "__main__":
    sys.exit(main())
