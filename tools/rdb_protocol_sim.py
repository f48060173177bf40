"""Developer tool (CPU): discrete-event model of the barrier protocol of csrc/conv3x3_rdb.cuh -- TMA producer, MMA
issuer, tensor pipe, two epilogue groups -- over the walk restated in tests/test_rdb_schedule.py.  Detects deadlocks
and out-of-protocol barrier use before any GPU time is spent.  Pair mode (simulate_pair): the CTA-pair form of
conv4 + conv5 -- two producers feeding the leader's landed barriers, count-8 drained / map-row barriers, multicast
commits, 14 stages, landed rings of 16 -- where every arrival also checks that it lands in the phase it is meant
for (a parity wait cannot tell a phase from the one two ahead).  python tools/rdb_protocol_sim.py"""
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


def simulate(nl, g, pieces, stages, verbose=False):
    ring = RINGS[nl]
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
        for (rnd, l, p, r, flush, n, seq) in steps:
            if flush:
                continue
            for _ in range(g):
                while not empty[stage].ready(phase ^ 1):
                    yield ("empty", stage)
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
                while not tdrain[l].ready((n - 1) & 1):
                    yield ("tdrain", l, n)
            if not flush:
                for _ in range(g):
                    k = fills % 8
                    while not lfull[l][k].ready((fills // 8) & 1):
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
            while not tfull[l].ready(n & 1):
                yield ("tfull", l, n)
            for _ in range(4):
                tdrain[l].arrive()
            if not real:
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

    if nl == 2:   # one producer and stage-ring slice per layer (conv3x3_rdb.cuh: rdb_layer_producer)
        ns0 = (stages + 1) // 2
        agents = {"producer0": layer_producer(0, 0, ns0), "producer1": layer_producer(1, ns0, stages - ns0)}
    else:
        agents = {"producer": producer()}
    for l in range(nl):
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


def simulate_pair(g, pieces2, stages, lring=16):
    """Two fused layers (conv4 + conv5) as a CTA pair; pieces2 = (rank 0's pieces, rank 1's pieces)."""
    nl = 2
    ring = RINGS[nl]
    steps2 = [list(walk(p, nl)) for p in pieces2]
    # both CTAs take the same walk: pieces, rows, flush steps (only b / x0 / the owned pixels differ)
    assert [s[:6] for s in steps2[0]] == [s[:6] for s in steps2[1]]
    pieces = pieces2[0]
    # leader: lfull (the leader's arrive.expect_tx + one load per CTA), tdrain / mfull (4 warps per CTA)
    lfull = [[Bar(3, f"lfull{l}.{s}") for s in range(lring)] for l in range(nl)]
    tdrain = [Bar(8, f"tdrain{l}") for l in range(nl)]
    mfull = [Bar(8, f"mfull0.{s}") for s in range(ring[0])]
    # per CTA: targets of the multicast commits
    empty = [[Bar(1, f"empty{s}@{c}") for s in range(stages)] for c in range(2)]
    tfull = [[Bar(1, f"tfull{l}@{c}") for l in range(nl)] for c in range(2)]
    mempty = [[Bar(1, f"mempty0.{s}@{c}") for s in range(ring[0])] for c in range(2)]
    lstage = [[[None] * lring for _ in range(nl)] for _ in range(2)]
    pipes = [deque() for _ in range(nl)]
    tma = deque()
    assert stages <= lring

    def producer(c):
        stage, phase, fill = 0, 0, 0
        fills = [0] * nl
        for (rnd, l, p, r, flush, n, seq) in steps2[c]:
            if flush:
                continue
            for _ in range(g):
                while not empty[c][stage].ready(phase ^ 1):
                    yield ("empty", c, stage)
                k = fills[l] % lring
                lstage[c][l][k] = stage
                if c == 0:
                    lfull[l][k].arrive(fills[l] // lring)  # arrive.expect_tx for both CTAs' bytes
                tma.append([3 + c, lfull[l][k], fills[l] // lring])
                fills[l] += 1
                fill += 1
                stage += 1
                if stage == stages:
                    stage, phase = 0, phase ^ 1

    def multicast(bars, phase):
        return ("commit", [(b, phase) for b in bars])

    def issuer(l):
        e = nl - 1 - l
        fills = 0
        for (p, r, flush, n, seq) in layer_steps(pieces, nl, l):
            pc = pieces[p]
            if n > 0:
                while not tdrain[l].ready((n - 1) & 1):
                    yield ("tdrain", l, n)
            if not flush:
                if l == 1:  # the in-CTA map first (NL == 2)
                    sq = seq[0] + (r - (pc["ra"] - (nl - 1)))
                    slot = sq % ring[0]
                    while not mfull[slot].ready((sq // ring[0]) & 1):
                        yield ("mfull", 0, sq)
                    pipes[l].append(("mma",))
                    pipes[l].append(multicast([mempty[0][slot], mempty[1][slot]], sq // ring[0]))
                for _ in range(g):
                    k = fills % lring
                    while not lfull[l][k].ready((fills // lring) & 1):
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
            while not tfull[c][l].ready(n & 1):
                yield ("tfull", c, l, n)
            for _ in range(4):
                tdrain[l].arrive(n)
            if not real or l == nl - 1:
                continue
            sq = seq[l] + (j - (pc["ra"] - e))
            slot = sq % ring[l]
            while not mempty[c][slot].ready(((sq // ring[l]) & 1) ^ 1):
                yield ("mempty", c, sq)
            for _ in range(4):
                mfull[slot].arrive(sq // ring[l])

    agents = {"producer0": producer(0), "producer1": producer(1)}
    for l in range(nl):
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
    sys.exit(0 if ok_all else 1)


if __name__ == "__main__":
    main()
