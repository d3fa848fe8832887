"""Model of the rotated bin walk of the decode kernels (csrc/decode_common.cuh): for every position on
the per-head task line, at which step do the CTAs that own that position for the different kv heads
process it? CPU only.

    python tools/decode_walk_sim.py [--batch 64] [--ctx 8192] [--heads 8] [--ctas 148]
                                    [--prefetch-distance D]

Prints the spread (max - min step over the heads) with and without the rotation. At the C2 shape the
rotation brings 95 % of the positions to spread 0 (the rest belong to bins that straddle a head
boundary); front to back the mean spread is ~190 steps of ~0.85 us.

With --prefetch-distance D it also models the page-wide L2 prefetch of the fp8 kernel: the CTA of
head (batch + tile) % heads prefetches a position when it loads the position D steps earlier in the
same segment of its walk (same task, consecutive tiles); at distance 0 it prefetches a tile just
before loading it itself. It reports the share of positions whose prefetch step is no later than
every consumer's load step, and by how many steps it leads.
"""
import argparse
import collections
import statistics


def walk(tb, heads, ctas, rotate, min_tiles=0):
    """For each CTA, the list of line positions x it loads, in walk order (drift-free: step = index)."""
    total = tb * heads
    p = max(-(-total // ctas), min_tiles)
    walks = []
    for i in range(ctas):
        x0 = i * p
        n = min(p, total - x0)
        if n <= 0:
            continue
        u0 = 0
        if rotate:
            u0 = (p - (x0 % tb) % p) % p
            if u0 >= n:
                u0 = 0
        walks.append([x0 + (u0 + t) % n for t in range(n)])
    return walks, p


def spreads(tb, heads, ctas, rotate, min_tiles=0):
    walks, p = walk(tb, heads, ctas, rotate, min_tiles)
    at = collections.defaultdict(list)
    for w in walks:
        for t, x in enumerate(w):
            at[x % tb].append(t)
    return [max(v) - min(v) for v in at.values()], p


def prefetch_leads(tb, tpr, heads, ctas, dist):
    """Per position on the per-head line: consumer-load step minus prefetch step (None: no prefetch)."""
    walks, _ = walk(tb, heads, ctas, True)
    load = collections.defaultdict(list)  # position -> load steps of its consumers
    pf = {}                               # position -> prefetch step of its duty CTA
    for w in walks:
        for t, x in enumerate(w):
            pos = x % tb
            load[pos].append(t)
            if t + dist < len(w):
                y = w[t + dist]
                # same segment: consecutive tiles of one task (one head's line, one request)
                if y == x + dist and y // tpr == x // tpr:
                    ypos = y % tb
                    if (y // tb) == (ypos // tpr + ypos % tpr) % heads:
                        pf[ypos] = t
    return [(min(load[pos]) - pf[pos]) if pos in pf else None for pos in range(tb)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--ctx", type=int, default=8192)
    ap.add_argument("--heads", type=int, default=8)
    ap.add_argument("--ctas", type=int, default=148)
    ap.add_argument("--prefetch-distance", type=int, default=None)
    a = ap.parse_args()
    tpr = -(-a.ctx // 128)
    tb = a.batch * tpr
    for rot in (False, True):
        s, p = spreads(tb, a.heads, a.ctas, rot)
        print(f"rotate={rot}: tiles/head {tb}, tiles/bin {p}: spread max {max(s)}, mean "
              f"{statistics.mean(s):.1f}, positions with spread 0: {sum(1 for v in s if v == 0) / len(s):.3f}")
    if a.prefetch_distance is not None:
        leads = prefetch_leads(tb, tpr, a.heads, a.ctas, a.prefetch_distance)
        have = [v for v in leads if v is not None]
        ahead = [v for v in have if v >= 0]
        print(f"prefetch distance {a.prefetch_distance}: positions prefetched {len(have) / tb:.3f}, "
              f"prefetched no later than every consumer's load {len(ahead) / tb:.3f}, lead over the "
              f"first consumer (steps): median {statistics.median(ahead) if ahead else 0}, "
              f"min {min(ahead) if ahead else 0}; at lead = distance "
              f"{sum(1 for v in ahead if v == a.prefetch_distance) / tb:.3f}")


if __name__ == "__main__":
    main()
