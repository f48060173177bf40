"""Developer tool (CPU): discrete-event model of the barrier protocol of csrc/conv3x3_rdb.cuh -- TMA producer, MMA
issuer, tensor pipe, two epilogue groups -- over the walk restated in tests/test_rdb_schedule.py.  Detects deadlocks
and out-of-protocol barrier use before any GPU time is spent.  Pair mode (simulate_pair): the CTA-pair form of
conv4 + conv5 -- two producers feeding the leader's landed barriers, count-8 drained / map-row barriers, multicast
commits, 14 stages, landed rings of 16 -- where every arrival also checks that it lands in the phase it is meant
for (a parity wait cannot tell a phase from the one two ahead).  The pair form of conv1..conv3 (simulate_pair, nl = 3)
reads x0 from a ring that each row enters once, and every wait checks its phase as well.  first_only (simulate and
simulate_pair, nl = 2): the conv4-only form (conv3x3_rdb_kernel<4, 2, PAIR, true>) -- the walk-order producer loads
conv4's chunks only, conv5's issuer and epilogue group do nothing and conv4's epilogue writes no map rows; its waits
check their phase too.  python tools/rdb_protocol_sim.py"""
import os
import sys
from collections import deque

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from test_rdb_schedule import RINGS, cta_pieces, tiles_x, walk  # noqa: E402
from test_rdb_pair_schedule import pair_pieces  # noqa: E402


class Bar:
    arrivals = 0  # all barriers: a tick in which anything arrived anywhere made progress

    def __init__(self, count, name):
        self.count, self.pending, self.phase, self.name = count, count, 0, name

    def arrive(self, phase=None):
        """phase: the phase this arrival belongs to (checked when given)"""
        assert phase is None or phase == self.phase, f"{self.name}: arrival for phase {phase} in phase {self.phase}"
        Bar.arrivals += 1
        self.pending -= 1
        if self.pending == 0:
            self.phase += 1
            self.pending = self.count

    def ready(self, parity):
        return (self.phase & 1) != parity

    def wait(self, use):
        """a parity wait for the completion of phase `use` (-1: the phase before the first, complete from the start);
        a parity cannot tell phase u from u + 2, so the barrier must be in phase use or use + 1 whenever it is polled"""
        assert use <= self.phase <= use + 1, f"{self.name}: waiting for phase {use} in phase {self.phase}"
        return self.ready(use & 1)


def layer_steps(pieces, nl, l):
    """What issuer l / epilogue group l iterate: their own layer only -- pieces in order, rows top to bottom, two
    flush steps per piece.  Yields (piece index, r, flush, n, seq[list: per map, of the piece's first row])."""
    e = nl - 1 - l
    n = 0
    seq = [0] * nl
    for p, pc in enumerate(pieces):
        for r in range(pc["ra"] - e - 1, pc["rb"] + e + 3):
            yield p, r, r > pc["rb"] + e, n, list(seq)
            n += 1
        for m in range(nl):
            seq[m] += (pc["rb"] - pc["ra"]) + 2 * (nl - 1 - m)


def simulate(nl, g, pieces, stages, verbose=False, first_only=False):
    assert not first_only or nl == 2
    ring = RINGS[nl]
    nact = 1 if first_only else nl   # layers whose issuer / epilogue group run

    def poll(bar, use):  # first_only: every wait also checks that it cannot pass a phase early
        return bar.wait(use) if first_only else bar.ready(use & 1)
    lfull = [[Bar(1, f"lfull{l}.{s}") for s in range(8)] for l in range(nl)]
    lstage = [[None] * 8 for _ in range(nl)]
    empty = [Bar(1, f"empty{s}") for s in range(stages)]
    tfull = [Bar(1, f"tfull{l}") for l in range(nl)]
    tdrain = [Bar(4, f"tdrain{l}") for l in range(nl)]
    mfull = [[Bar(4, f"mfull{m}.{s}") for s in range(max(ring[m], 1))] for m in range(nl - 1)]
    mempty = [[Bar(1, f"mempty{m}.{s}") for s in range(max(ring[m], 1))] for m in range(nl - 1)]
    pipes = [deque() for _ in range(nl)]   # per issuing thread: its MMAs complete in order; a commit follows them
    tma = deque()                          # in-flight loads: [ticks left, bar]
    steps = list(walk(pieces, nl))
    # the per-layer iteration must be the walk restricted to the layer
    for l in range(nl):
        assert [(p, r, fl, n) for (_, ll, p, r, fl, n, _) in steps if ll == l] == [(p, r, fl, n) for (p, r, fl, n, _) in
                                                                                 layer_steps(pieces, nl, l)]
        assert [sq for (_, ll, p, r, fl, n, sq) in steps if ll == l] == [sq for (p, r, fl, n, sq) in layer_steps(pieces, nl, l)]

    def producer():
        stage, phase = 0, 0
        fills = [0] * nl
        fill = 0
        for (rnd, l, p, r, flush, n, seq) in steps:
            if flush or l >= nact:
                continue
            for _ in range(g):
                while not poll(empty[stage], fill // stages - 1):
                    yield ("empty", stage)
                fill += 1
                k = fills[l] % 8
                fills[l] += 1
                lstage[l][k] = stage
                tma.append([3, lfull[l][k]])
                stage += 1
                if stage == stages:
                    stage, phase = 0, phase ^ 1
        return

    def issuer(l):
        e = nl - 1 - l
        fills = 0
        for (p, r, flush, n, seq) in layer_steps(pieces, nl, l):
            pc = pieces[p]
            if n > 0:
                while not poll(tdrain[l], n - 1):
                    yield ("tdrain", l, n)
            if not flush:
                for _ in range(g):
                    k = fills % 8
                    while not poll(lfull[l][k], fills // 8):
                        yield ("lfull", l, fills)
                    st = lstage[l][k]
                    fills += 1
                    pipes[l].append(("mma",))
                    pipes[l].append(("commit", empty[st]))
                for m in range(nl - 1):
                    if m < l:
                        sq = seq[m] + (r - (pc["ra"] - (nl - 1 - m)))
                        slot = sq % ring[m]
                        while not mfull[m][slot].ready((sq // ring[m]) & 1):
                            yield ("mfull", m, sq)
                        pipes[l].append(("mma",))
                        if l == nl - 1 or r < pc["ra"] - e or r > pc["rb"] + e - 1:
                            pipes[l].append(("commit", mempty[m][slot]))
            pipes[l].append(("commit", tfull[l]))
        return

    def epilogue(l):
        e = nl - 1 - l
        for (p, r, flush, n, seq) in layer_steps(pieces, nl, l):
            pc = pieces[p]
            j = r - 1
            real = pc["ra"] - e <= j < pc["rb"] + e
            while not poll(tfull[l], n):
                yield ("tfull", l, n)
            for _ in range(4):
                tdrain[l].arrive()
            if not real or first_only:
                continue
            if l < nl - 1:
                sq = seq[l] + (j - (pc["ra"] - e))
                slot = sq % ring[l]
                while not mempty[l][slot].ready(((sq // ring[l]) & 1) ^ 1):
                    yield ("mempty", l, sq)
                for _ in range(4):
                    mfull[l][slot].arrive()
        return

    def layer_producer(l, s0, ns):
        idx, phase, fills = 0, 0, 0
        for (p, r, flush, n, seq) in layer_steps(pieces, nl, l):
            if flush:
                continue
            for _ in range(g):
                stage = s0 + idx
                while not empty[stage].ready(phase ^ 1):
                    yield ("empty", stage)
                k = fills % 8
                fills += 1
                lstage[l][k] = stage
                tma.append([3, lfull[l][k]])
                idx += 1
                if idx == ns:
                    idx, phase = 0, phase ^ 1
        return

    if nl == 2 and not first_only:   # one producer and stage-ring slice per layer (conv3x3_rdb.cuh: rdb_layer_producer)
        ns0 = (stages + 1) // 2
        agents = {"producer0": layer_producer(0, 0, ns0), "producer1": layer_producer(1, ns0, stages - ns0)}
    else:
        agents = {"producer": producer()}
    for l in range(nact):
        agents[f"issuer{l}"] = issuer(l)
        agents[f"epi{l}"] = epilogue(l)
    blocked = {}
    ticks = 0
    while agents:
        progressed = False
        seen = Bar.arrivals
        for name in list(agents):
            try:
                blocked[name] = next(agents[name])
            except StopIteration:
                del agents[name]
                blocked.pop(name, None)
                progressed = True
        for pipe in pipes:   # each thread's ops complete in its own order, one per tick
            if pipe:
                op = pipe.popleft()
                if op[0] == "commit":
                    op[1].arrive()
                progressed = True
        for t in list(tma):
            t[0] -= 1
            if t[0] <= 0:
                t[1].arrive()
                tma.remove(t)
            progressed = True
        ticks += 1
        progressed = progressed or Bar.arrivals != seen
        if not progressed and not any(pipes) and not tma:
            return False, dict(blocked)
        if ticks > 5_000_000:
            return False, {"timeout": dict(blocked)}
    return True, ticks


def simulate_pair(g, pieces2, stages, lring=16, nl=2, first_only=False):
    """The CTA-pair forms; pieces2 = (rank 0's pieces, rank 1's pieces).  nl = 2: conv4 + conv5 (G = 4) -- the
    walk-order stage ring, per-layer landed rings of `lring`.  nl = 3: conv1..conv3 (G = 1) -- the x0 ring of `stages`
    row tiles, each x0 row loaded once and released by its last reader.  Every wait checks that the barrier is in the
    phase it waits for or the one after it (a parity wait passes early on the phase before it and never passes two
    phases after it); every arrival checks that it lands in the phase it is meant for."""
    xring = nl == 3
    assert not xring or g == 1
    assert not first_only or nl == 2
    nact = 1 if first_only else nl   # layers whose issuer / epilogue groups run
    ring = RINGS[nl]
    steps2 = [list(walk(p, nl)) for p in pieces2]
    # both CTAs take the same walk: pieces, rows, flush steps (only b / x0 / the owned pixels differ)
    assert [s[:6] for s in steps2[0]] == [s[:6] for s in steps2[1]]
    pieces = pieces2[0]
    # leader: full barriers (the leader's arrive.expect_tx + one load per CTA), tdrain / mfull (4 warps per CTA)
    lfull = [[Bar(3, f"lfull{l}.{s}") for s in range(lring)] for l in range(nl)]
    xfull = [Bar(3, f"xfull{s}") for s in range(stages)]
    tdrain = [Bar(8, f"tdrain{l}") for l in range(nl)]
    mfull = [[Bar(8, f"mfull{m}.{s}") for s in range(ring[m])] for m in range(nl - 1)]
    # per CTA: targets of the multicast commits
    empty = [[Bar(1, f"empty{s}@{c}") for s in range(stages)] for c in range(2)]
    tfull = [[Bar(1, f"tfull{l}@{c}") for l in range(nl)] for c in range(2)]
    mempty = [[[Bar(1, f"mempty{m}.{s}@{c}") for s in range(ring[m])] for m in range(nl - 1)] for c in range(2)]
    lstage = [[[None] * lring for _ in range(nl)] for _ in range(2)]
    xrow = [[None] * stages for _ in range(2)]   # (piece, row) each CTA's x0 ring slot holds
    xbase = [0]                                  # x0 ring: sequence number of each piece's first row, ra - nl
    for pc in pieces:
        xbase.append(xbase[-1] + (pc["rb"] - pc["ra"]) + 2 * nl)
    pipes = [deque() for _ in range(nl)]
    tma = deque()
    assert stages <= lring

    def latency(c, k):  # loads land out of order
        return 3 + c + (5 * k) % 7

    def producer(c):
        stage, phase, fill = 0, 0, 0
        fills = [0] * nl
        for (rnd, l, p, r, flush, n, seq) in steps2[c]:
            if flush or l >= nact:
                continue
            for _ in range(g):
                while not empty[c][stage].wait(fill // stages - 1):
                    yield ("empty", c, stage)
                k = fills[l] % lring
                lstage[c][l][k] = stage
                if c == 0:
                    lfull[l][k].arrive(fills[l] // lring)  # arrive.expect_tx for both CTAs' bytes
                tma.append([latency(c, fill), lfull[l][k], fills[l] // lring])
                fills[l] += 1
                fill += 1
                stage += 1
                if stage == stages:
                    stage, phase = 0, phase ^ 1

    def x0_producer(c):
        sq = 0
        for p, pc in enumerate(pieces2[c]):
            for r in range(pc["ra"] - nl, pc["rb"] + nl):
                slot = sq % stages
                while not empty[c][slot].wait(sq // stages - 1):
                    yield ("empty", c, slot)
                xrow[c][slot] = (p, r)
                if c == 0:
                    xfull[slot].arrive(sq // stages)  # arrive.expect_tx for both CTAs' bytes
                tma.append([latency(c, sq), xfull[slot], sq // stages])
                sq += 1

    def multicast(bars, phase):
        return ("commit", [(b, phase) for b in bars])

    def issuer(l):
        e = nl - 1 - l
        fills = 0
        for (p, r, flush, n, seq) in layer_steps(pieces, nl, l):
            pc = pieces[p]
            if n > 0:
                while not tdrain[l].wait(n - 1):
                    yield ("tdrain", l, n)
            if not flush:
                # K order: two fused layers take the in-CTA map first, three take x0 first
                for kind in (("map", "global") if nl == 2 else ("global", "map")):
                    if kind == "map":
                        for m in range(l):
                            sq = seq[m] + (r - (pc["ra"] - (nl - 1 - m)))
                            slot = sq % ring[m]
                            while not mfull[m][slot].wait(sq // ring[m]):
                                yield ("mfull", m, sq)
                            pipes[l].append(("mma",))
                            if l == nl - 1 or r < pc["ra"] - e or r > pc["rb"] + e - 1:
                                pipes[l].append(multicast([mempty[0][m][slot], mempty[1][m][slot]], sq // ring[m]))
                    elif xring:
                        if r == pc["ra"] - e - 1:
                            # a piece's first step follows flush steps: before the row can be given back, the layers
                            # before this one must have read it -- their map rows r are written (their steps on r + 1)
                            for m in range(l):
                                sq = seq[m] + (r - (pc["ra"] - (nl - 1 - m)))
                                while not mfull[m][sq % ring[m]].wait(sq // ring[m]):
                                    yield ("mfull", m, sq)
                        sq = xbase[p] + (r - (pc["ra"] - nl))
                        slot = sq % stages
                        while not xfull[slot].wait(sq // stages):
                            yield ("xfull", l, sq)
                        assert xrow[0][slot] == xrow[1][slot] == (p, r), (l, p, r, xrow[0][slot], xrow[1][slot])
                        pipes[l].append(("mma",))
                        # the last layer that reads the row gives the slot back
                        if l == nl - 1 or r < pc["ra"] - e or r > pc["rb"] + e - 1:
                            pipes[l].append(multicast([empty[0][slot], empty[1][slot]], sq // stages))
                    else:
                        for _ in range(g):
                            k = fills % lring
                            while not lfull[l][k].wait(fills // lring):
                                yield ("lfull", l, fills)
                            st = lstage[0][l][k]
                            assert lstage[1][l][k] == st, "the CTAs of a pair loaded a chunk into different stages"
                            fills += 1
                            pipes[l].append(("mma",))
                            pipes[l].append(("commit_stage", st))
            pipes[l].append(multicast([tfull[0][l], tfull[1][l]], n))

    stage_commits = [0] * stages

    def epilogue(c, l):
        e = nl - 1 - l
        for (p, r, flush, n, seq) in layer_steps(pieces2[c], nl, l):
            pc = pieces2[c][p]
            j = r - 1
            real = pc["ra"] - e <= j < pc["rb"] + e
            while not tfull[c][l].wait(n):
                yield ("tfull", c, l, n)
            for _ in range(4):
                tdrain[l].arrive(n)
            if not real or l == nl - 1 or first_only:
                continue
            sq = seq[l] + (j - (pc["ra"] - e))
            slot = sq % ring[l]
            while not mempty[c][l][slot].wait(sq // ring[l] - 1):
                yield ("mempty", c, l, sq)
            for _ in range(4):
                mfull[l][slot].arrive(sq // ring[l])

    agents = {f"producer{c}": (x0_producer(c) if xring else producer(c)) for c in range(2)}
    for l in range(nact):
        agents[f"issuer{l}"] = issuer(l)
        for c in range(2):
            agents[f"epi{l}@{c}"] = epilogue(c, l)
    blocked = {}
    ticks = 0
    while agents:
        progressed = False
        seen = Bar.arrivals
        for name in list(agents):
            try:
                blocked[name] = next(agents[name])
            except StopIteration:
                del agents[name]
                blocked.pop(name, None)
                progressed = True
        for pipe in pipes:
            if pipe:
                op = pipe.popleft()
                if op[0] == "commit":
                    for b, ph in op[1]:
                        b.arrive(ph)
                elif op[0] == "commit_stage":
                    st = op[1]
                    for c in range(2):
                        empty[c][st].arrive(stage_commits[st])
                    stage_commits[st] += 1
                progressed = True
        for t in list(tma):
            t[0] -= 1
            if t[0] <= 0:
                t[1].arrive(t[2])
                tma.remove(t)
            progressed = True
        ticks += 1
        progressed = progressed or Bar.arrivals != seen
        if not progressed and not any(pipes) and not tma:
            return False, dict(blocked)
        if ticks > 5_000_000:
            return False, {"timeout": dict(blocked)}
    return True, ticks


def main():
    cases = [(3, 1, 1, 4, 16, 4), (2, 4, 1, 4, 16, 4), (3, 1, 2, 24, 40, 48), (2, 4, 2, 24, 40, 48), (3, 1, 64, 208, 416, 148),
             (2, 4, 64, 208, 416, 148), (3, 1, 3, 5, 70, 5), (2, 4, 3, 5, 70, 5)]
    ok_all = True
    for nl, g, batch, band_h, width, grid in cases:
        ntx = tiles_x(width, nl)
        grid = min(grid, batch * ntx * band_h)
        stages = 5 if nl == 3 else 5
        for cta in sorted(set([0, 1, grid // 2, grid - 1])):
            pieces = cta_pieces(cta, grid, batch, band_h, width, nl)
            ok, info = simulate(nl, g, pieces, stages)
            print(f"NL={nl} G={g} batch={batch} band_h={band_h} W={width} grid={grid} cta={cta}: "
                  f"{'ok, ticks ' + str(info) if ok else 'DEADLOCK ' + str(info)}")
            ok_all &= ok
    # CTA pairs: conv4 + conv5, 14 stages; batch 1 has an odd column count (a phantom column on rank 1)
    for batch, band_h, width, grid in [(1, 4, 416, 148), (3, 20, 416, 148), (64, 208, 416, 148), (1, 208, 416, 148),
                                       (3, 4, 200, 148), (2, 9, 64, 13 * 2)]:
        ntx = tiles_x(width, 2)
        pairs = min(grid // 2, (batch * ntx + 1) // 2 * band_h)
        for u in sorted(set([0, 1, pairs // 2, pairs - 1])):
            pcs = [pair_pieces(2 * u + rank, 2 * pairs, batch, band_h, width, 2) for rank in (0, 1)]
            ok, info = simulate_pair(4, pcs, 14)
            print(f"pair NL=2 G=4 batch={batch} band_h={band_h} W={width} pairs={pairs} pair={u}: "
                  f"{'ok, ticks ' + str(info) if ok else 'DEADLOCK ' + str(info)}")
            ok_all &= ok
    # CTA pairs: conv1..conv3 with the x0 ring (11 rows; 4, the launcher's minimum); band_h 4 and 5: pieces shorter
    # than the ring, whose edge rows the later layers skip
    for batch, band_h, width, grid in [(1, 4, 416, 148), (3, 20, 416, 148), (64, 208, 416, 148), (1, 208, 416, 148),
                                       (3, 5, 200, 148), (2, 9, 64, 13 * 2), (3, 4, 416, 4)]:
        ntx = tiles_x(width, 3)
        pairs = min(grid // 2, (batch * ntx + 1) // 2 * band_h)
        for u in sorted(set([0, 1, pairs // 2, pairs - 1])):
            pcs = [pair_pieces(2 * u + rank, 2 * pairs, batch, band_h, width, 3) for rank in (0, 1)]
            for xr in (11, 4):
                ok, info = simulate_pair(1, pcs, xr, nl=3)
                print(f"pair NL=3 G=1 x0 ring {xr} batch={batch} band_h={band_h} W={width} pairs={pairs} pair={u}: "
                      f"{'ok, ticks ' + str(info) if ok else 'DEADLOCK ' + str(info)}")
                ok_all &= ok
    # the conv4-only form: single CTAs with the launcher's 8 stages, pairs with 16; batch 1 has a phantom column
    for batch, band_h, width, grid in [(1, 208, 416, 148), (16, 208, 416, 148), (64, 208, 416, 148), (3, 4, 200, 148),
                                       (2, 9, 64, 13 * 2)]:
        ntx = tiles_x(width, 2)
        g1 = min(grid, batch * ntx * band_h)
        for cta in sorted(set([0, 1, g1 // 2, g1 - 1])):
            ok, info = simulate(2, 4, cta_pieces(cta, g1, batch, band_h, width, 2), 8, first_only=True)
            print(f"conv4-only NL=2 G=4 batch={batch} band_h={band_h} W={width} grid={g1} cta={cta}: "
                  f"{'ok, ticks ' + str(info) if ok else 'DEADLOCK ' + str(info)}")
            ok_all &= ok
        pairs = min(grid // 2, (batch * ntx + 1) // 2 * band_h)
        for u in sorted(set([0, 1, pairs // 2, pairs - 1])):
            pcs = [pair_pieces(2 * u + rank, 2 * pairs, batch, band_h, width, 2) for rank in (0, 1)]
            ok, info = simulate_pair(4, pcs, 16, first_only=True)
            print(f"conv4-only pair NL=2 G=4 batch={batch} band_h={band_h} W={width} pairs={pairs} pair={u}: "
                  f"{'ok, ticks ' + str(info) if ok else 'DEADLOCK ' + str(info)}")
            ok_all &= ok
    sys.exit(0 if ok_all else 1)


if __name__ == "__main__":
    main()
