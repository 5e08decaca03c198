"""Per-unit timeline of CTA 0 of the tcgen05 tiled pass (NMFK_TC_TRACE): cycles between the stamps of the quotient
warp, the MMA issuers and the loading warp (a stager warp in the first generation).  usage: tc_trace.py n m k R  (runs one
solve, prints the tables)"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "nmfk.jl_b200", "python"))
os.environ["NMFK_TC_TRACE"] = "/tmp/tc_trace.bin"
import numpy as np  # noqa: E402
import nmfk_b200 as nb  # noqa: E402
from nmfk_b200 import synth  # noqa: E402

n, m, k, R = (int(v) for v in sys.argv[1:5])
with nb.Context(0) as ctx:
    ctx.set_X(synth.mixture(n, m, 8, seed=3, dtype=np.float32))
    for it in (2, 2):  # the second solve is warm
        b = ctx.batch(k, R)
        b.init_random(1)
        ctx.solve([b], nb.default_params(maxiter=it, engine=2))
        b.close()
t = np.fromfile("/tmp/tc_trace.bin", dtype=np.int64).reshape(3, 64, 8)
t0 = t[t > 0].min()
q, mm, st = t[0], t[1], t[2]
if os.environ.get("NMFK_TC_GEN", "2") != "1":
    print("gen2 quotient detail (group 0): unit | pwait ldP half0 afullwait drain+st0 half1+st1 arrive | cycle")
    for u in range(8, 40, 2):
        qq = q[u]
        if qq[0] == 0 or q[u + 2, 0] == 0:
            break
        print("%4d | %6d %5d %6d %6d %6d %6d %6d | %6d" % (u, qq[1] - qq[0], qq[2] - qq[1], qq[5] - qq[2], qq[6] - qq[5], qq[7] - qq[6],
                                                         qq[3] - qq[7], qq[4] - qq[3], q[u + 2, 0] - qq[0]))
if os.environ.get("NMFK_TC_GEN", "2") == "1":
    print("unit | quotient group 0 (even units): pwait  ld  compute+drain  st+arrive | cycle of 2 units || mma (this unit): qwait mma2-issue vwait mma1-issue || stager: cpwait vempty convert")
    for u in range(8, 40, 2):
        if q[u, 0] == 0 or q[u + 2, 0] == 0:
            break
        qq = q[u]
        print("%4d | %6d %5d %6d %8d | %6d || %6d %6d %6d %6d || %6d %6d %6d   (q start @%d, mma2 @%d)" % (
            u, qq[1] - qq[0], qq[2] - qq[1], qq[3] - qq[2], qq[4] - qq[3], q[u + 2, 0] - qq[0],
            mm[u, 1] - mm[u, 0], mm[u, 2] - mm[u, 1], mm[u, 4] - mm[u, 3], mm[u, 5] - mm[u, 4],
            st[u, 1] - st[u - 1, 0], st[u, 2] - st[u, 1], st[u, 3] - st[u, 2], qq[0] - t0, mm[u, 0] - t0))
    sys.exit(0)


def d(a, b):  # a - b, "-" where either stamp was not taken
    return "%6d" % (a - b) if a > 0 and b > 0 else "%6s" % "-"


# q_full(u) arrive = the quotient warp's stamp after its arrive (0, u, 4); MMA#2 thread: reaches u (1, u, 0), has seen q_full
# (1, u, 1), has issued and committed (1, u, 2); the group sees a_full(u) at (0, u + 2, 6)
print("unit | q_full(u) @ | MMA#2 reaches u: @  late by | qwait | q_full seen - q_full | issue | a_full seen - MMA#2 issued | group a_full wait | cycle of 2 units")
for u in range(8, 40, 2):
    if q[u, 0] == 0 or q[u + 2, 0] == 0:
        break
    print("%4d | %11d | %18d %8d | %5s | %20s | %5s | %27s | %17s | %6d" % (
        u, q[u, 4] - t0, mm[u, 0] - t0, mm[u, 0] - q[u, 4], d(mm[u, 1], mm[u, 0]), d(mm[u, 1], q[u, 4]), d(mm[u, 2], mm[u, 1]), d(q[u + 2, 6], mm[u, 2]),
        d(q[u + 2, 6], q[u + 2, 5]), q[u + 2, 0] - q[u, 0]))
# loading, per unit: v_empty wait, V bulk copy, x_empty wait, X loads (role 2).  The last two columns are written only by the
# kernel before the load warp, where the MMA#2 thread also loaded, with profiles/r05_main_stamps.diff applied: its loop top
# (1, u, 6) -> reaching u (1, u, 0), and the mbar_test polls and opportunistic loads after the issue (1, u, 2) -> (2, u, 3)
print("unit | vwait load_v | xwait load_x | MMA#2 thread: loop top -> reaches u, post-issue polls")
for u in range(8, 40):
    if mm[u, 0] == 0:
        break
    print("%4d | %6s %6s | %6s %6s | %6s %6s" % (u, d(st[u, 1], st[u, 0]), d(st[u, 2], st[u, 1]), d(st[u, 5], st[u, 4]),
                                                   d(st[u, 6], st[u, 5]), d(mm[u, 0], mm[u, 6]), d(st[u, 3], mm[u, 2])))
