"""Shared-memory wavefronts of rk_fhn_tile_kernel (csrc/rk.cu) per warp and RK stage, replayed from its addresses.

Runs on the CPU.  For every shared-memory instruction of one stage (the plain form, SHX = false) the script forms each
thread's byte address exactly as the kernel does and counts the wavefronts under the bank model of the SM: 32 banks of
4 bytes; a 64-bit access is served in two half-warp phases and a 128-bit access in four quarter-warp phases; within a
phase the wavefront count is the largest number of distinct 4-byte words any one bank has to deliver (threads reading
the same word share it).  Two orders of the left / right column loads are compared:

  plain      every thread loads its left neighbour column, then its right one (the kernel before the change);
  alternate  threads whose block row has flip set load the right neighbour first (the kernel now), so one
             instruction reads odd and even columns in the two halves of a half-warp.

Per (c, r) the kernel issues one 128-bit store of its own pair, one 128-bit load each of the pair above and below, and
two 64-bit column loads; the floor is one wavefront per phase (a phase moves at most 128 bytes).

usage: python scripts/rk_shared_wavefronts.py [--dx 4 6 8 12 16 18 20 32]
"""
import argparse


def thread_setup(t, dx, TY):
    hx = dx // 2
    ntile = hx * (dx // TY)
    tt = t if t < ntile else 0
    ix0, iy0 = 2 * (tt % hx), TY * (tt // hx)
    yu = (dx if iy0 == 0 else iy0) - 1
    yd = 0 if iy0 + TY == dx else iy0 + TY
    xl = (dx if ix0 == 0 else ix0) - 1
    xr = 0 if ix0 + 2 == dx else ix0 + 2
    flip = ((iy0 // TY) ^ (ix0 >> 4)) & 1
    return dict(active=t < ntile, o00=iy0 * dx + ix0, oup=yu * dx + ix0, odn=yd * dx + ix0,
                ol=iy0 * dx + xl, orr=iy0 * dx + xr, flip=flip)


def wavefronts(addrs, width):
    """addrs: byte addresses of the 32 lanes (None = lane does not access); width 8 or 16 bytes.
    Returns (wavefronts, floor): a phase moves at most 128 bytes, so the floor is one per phase with an access."""
    phase = 16 if width == 8 else 8
    total = floor = 0
    for p0 in range(0, 32, phase):
        words = {}
        for a in addrs[p0:p0 + phase]:
            if a is None:
                continue
            for w in range(a // 4, (a + width) // 4):
                words.setdefault(w % 32, set()).add(w)
        total += max((len(s) for s in words.values()), default=0)
        floor += 1 if words else 0
    return total, floor


def stage_cost(dx, TY, order):
    npts = dx * dx
    threads = ((npts // (2 * TY) + 31) // 32) * 32
    T = [thread_setup(t, dx, TY) for t in range(threads)]
    cost = floor = 0
    for par in (0, 1):  # the two stage buffers alternate: report their mean
        for w0 in range(0, threads, 32):
            lanes = T[w0:w0 + 32]
            for c in range(2):
                base = par * 2 * npts + c * npts
                ins = []
                for r in range(TY):
                    ins += [([8 * (base + x["o00"] + r * dx) if x["active"] else None for x in lanes], 16)]
                    if order == "plain":
                        first = [x["ol"] for x in lanes]
                        second = [x["orr"] for x in lanes]
                    else:
                        first = [x["orr"] if x["flip"] else x["ol"] for x in lanes]
                        second = [x["ol"] if x["flip"] else x["orr"] for x in lanes]
                    ins += [([8 * (base + o + r * dx) for o in first], 8), ([8 * (base + o + r * dx) for o in second], 8)]
                ins += [([8 * (base + x["oup"]) for x in lanes], 16), ([8 * (base + x["odn"]) for x in lanes], 16)]
                for a, wd in ins:
                    wf, fl = wavefronts(a, wd)
                    cost += wf
                    floor += fl
    warps = threads // 32
    return cost / (2 * warps), floor / (2 * warps), warps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dx", type=int, nargs="*", default=[4, 6, 8, 12, 16, 18, 20, 32])
    args = ap.parse_args()
    print("# rk_fhn_tile_kernel, shared-memory wavefronts per warp and RK stage (mean over warps and both stage buffers)")
    print(f"# {'d_x':>4} {'TY':>3} {'warps':>5} {'plain':>7} {'alternate':>9} {'floor':>6}")
    for dx in args.dx:
        for TY in (2, 1):
            if dx % 2 or dx % TY:
                continue
            old, floor, warps = stage_cost(dx, TY, "plain")
            new, _, _ = stage_cost(dx, TY, "alternate")
            print(f"  {dx:>4} {TY:>3} {warps:>5} {old:>7.1f} {new:>9.1f} {floor:>6.1f}")


if __name__ == "__main__":
    main()
