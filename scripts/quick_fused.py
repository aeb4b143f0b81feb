"""Development aid: time the batched fused step (cfg3 shape) and check a few filters against the oracle.

    python scripts/quick_fused.py [--filters 65536] [--landmarks 20] [--steps 10] [--warmup 3] [--unknown] [--check 8]

n = 20 runs the tile kernel on the cfg3 world (the shape bench.py times); any other n <= 64 runs the staircase kernel on
a grid of n landmarks that are all in sight.

Not part of the product or of bench.py; it exists so that a kernel change can be judged in one short GPU run.
"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def world(tg, n):
    if n == 20:
        return tg.dense_world(n)
    # dense_world's rejection sampling cannot place much more than 40 tubes
    nx = int(np.ceil(np.sqrt(n)))
    w = tg.grid_world(nx, -(-n // nx), pitch=0.3, n_slots=n, max_visible=3.0)
    w.tubes_x, w.tubes_y = w.tubes_x[:n], w.tubes_y[:n]
    return w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--filters", type=int, default=65536)
    ap.add_argument("--landmarks", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--check", type=int, default=8)
    ap.add_argument("--unknown", action="store_true")
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()
    import torch

    import ekf_slam_ml_b200 as pkg
    from _oracle import OracleEKF, sigma_err, state_err

    tg = pkg.tracegen
    B, n, T = a.filters, a.landmarks, a.steps + a.warmup
    t0 = time.time()
    if a.unknown:
        M = 12
        tr = tg.simulate_unknown(world(tg, n), B, T, seed=4242, m_max=M)
        d_tw = torch.from_numpy(np.ascontiguousarray(tr["twists"])).cuda()
        d_me = torch.from_numpy(np.ascontiguousarray(tr["meas"])).cuda()
        d_ct = torch.from_numpy(np.ascontiguousarray(tr["count"])).cuda()
    else:
        tr = tg.simulate_known(world(tg, n), B, T + 1, seed=2026, workers=os.cpu_count())
        d_tw = torch.from_numpy(np.ascontiguousarray(tr["twists"])).cuda()
        d_xy = torch.from_numpy(np.ascontiguousarray(tr["xy"])).cuda()
        d_vis = torch.from_numpy(np.ascontiguousarray(tr["vis"])).cuda()
    print(f"traces: {time.time() - t0:.1f} s", flush=True)
    torch.cuda.synchronize()
    best = None
    for rep in range(a.repeat):
        bt = pkg.EKFBatch(B, n)

        def step(t):
            if a.unknown:
                bt.step_unknown_dev(d_tw[t].data_ptr(), d_me[t].data_ptr(), d_ct[t].data_ptr(), M)
            else:
                bt.step_known_dev(d_tw[t].data_ptr(), d_xy[t].data_ptr(), d_vis[t].data_ptr())

        T0 = 0 if a.unknown else 1
        if not a.unknown:
            step(0)  # the node's init-only call
        for t in range(T0, T0 + a.warmup):
            step(t)
        bt.sync()
        u0 = bt.update_count
        L = pkg._lib.load()
        prof = hasattr(L, "ekf_debug_tile_prof") if os.environ.get("EKF_B200_LIB") else False
        if prof:
            import ctypes
            buf = (ctypes.c_uint64 * 16)()
            L.ekf_debug_tile_prof(buf)
        bt.timer_start()
        for t in range(T0 + a.warmup, T0 + T):
            step(t)
        ms = bt.timer_stop()
        upd = bt.update_count - u0
        if prof:
            L.ekf_debug_tile_prof(buf)
            tot = float(sum(buf))
            names = ["inputs", "wait landing", "regs+predict", "meas entry", "corr (rest)", "write-back", "-", "loop top",
                     "gain_w A", "gain_k A", "robcols+H_j B", "gain_w B", "gain_k B", "last pass", "H_j A' || pass", "stage+gather"]
            if a.unknown:
                names[8:] = ["mirrors", "distances", "argmin+gates", "creation", "H_j+gather", "gain_w", "gain_k", "pass+stage"]
            print("   phase cycles per filter-step: " + ", ".join(
                f"{n_} {buf[k] / (a.steps * B):.0f} ({100 * buf[k] / tot:.0f}%)" for k, n_ in enumerate(names) if buf[k]))
        print(f"rep {rep}: {ms / a.steps:.4f} ms/step, {upd / a.steps / B:.2f} upd/filter-step, "
              f"{upd / (ms * 1e-3):.4e} upd/s", flush=True)
        best = ms if best is None else min(best, ms)
        if rep + 1 < a.repeat:
            bt.close()
    # parity of the last repetition
    states = bt.states()
    rng = np.random.default_rng(0)
    worst = 0.0
    for b in sorted(set([0, B - 1] + list(rng.integers(0, B, a.check)))):
        o = OracleEKF(n)
        if a.unknown:
            known = np.zeros(n, np.uint8)
            for t in range(T):
                o.prediction(*tr["twists"][t, b])
                o.data_association(tr["meas"][t, b, :tr["count"][t, b]], known)
        else:
            for t in range(T + 1):
                o.prediction(*tr["twists"][t, b])
                o.measurement(tr["xy"][t, b], tr["vis"][t, b])
        e = max(state_err(states[b], o.state), sigma_err(bt.sigma(int(b)), o.sigma))
        worst = max(worst, e)
    print(f"parity: worst scaled error over checked filters {worst:.3e} ({'OK' if worst < 1e-9 else 'FAIL'})")
    bt.close()
    sys.exit(0 if worst < 1e-9 else 1)


if __name__ == "__main__":
    main()
