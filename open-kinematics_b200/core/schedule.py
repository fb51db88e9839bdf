"""Phase assignment of the left-looking contributions of the block factorisation and the triangular
solves.

The kernel walks the elimination-tree levels one warp phase at a time.  A contribution to a destination
(a block row of the factor, a carried right-hand side, a column of a triangular solve) may run in any
phase after the one that finalises its source column and no later than the phase that finalises the
destination.  Running every contribution in its destination's own phase leaves the trunk of the tree
(a few columns per level, long gather lists) to a handful of lanes while the lanes of the early levels
idle; this module spreads the contributions over the phases they may run in.

Cost model (shared-memory wavefronts, the pipe the kernel is bound by): the tasks of a phase are taken
round-robin by 32 lanes, heaviest first.  Every trip of a round's gather loop costs 12 64-bit loads per
active half-warp plus one table word; every task visit costs 6 loads / stores of the destination per
half-warp plus 3 table words, and a visit that finalises a solve column 6 more loads of the diagonal
factor per half-warp.

Within a task the contributions keep the order of the destination's list; a destination visited in
several phases sums its contributions phase by phase, so results change only in the rounding.
"""

from __future__ import annotations

from dataclasses import dataclass

LANES = 32
HALF = 16


@dataclass
class Dest:
    """One destination: ``weight`` tasks (the three rows of a factor block) that share the contribution
    list; contribution ``c`` may run in phases ``lo[c] .. home``; ``final`` = the home phase always
    visits the destination (a solve column is finalised there even without contributions)."""
    weight: int
    home: int
    lo: list
    final: bool = False


def phase_cost(tasks) -> int:
    """Modelled wavefronts of one phase; ``tasks`` = ``(n_contributions, finalises)`` per lane task."""
    return _sorted_cost(sorted(tasks, key=lambda t: -t[0]))


def _sorted_cost(order) -> int:
    cost = 0
    for r0 in range(0, len(order), LANES):
        rnd = order[r0:r0 + LANES]
        for h0 in (0, HALF):
            half = rnd[h0:h0 + HALF]
            if half:
                cost += 6 + 6 * any(fin for _, fin in half)
        cost += 3
        n_active = len(rnd)
        for q in range(rnd[0][0]):
            while rnd[n_active - 1][0] <= q:
                n_active -= 1
            cost += 12 * (1 if n_active <= HALF else 2) + 1
    return cost


def _hist_cost(hist: dict) -> int:
    """``phase_cost`` of a phase given as ``{(n_contributions, finalises): lane tasks}``."""
    order = []
    for key in sorted(hist, key=lambda k: (-k[0], not k[1])):
        order += [key] * hist[key]
    return _sorted_cost(order)


class _State:
    """Per phase a histogram of its lane tasks, and which destinations visit it with how many
    contributions."""

    def __init__(self, dests: list, phases: list, n_phases: int):
        self.dests = dests
        self.count = [dict() for _ in range(n_phases)]
        for d, ph in enumerate(phases):
            for p in ph:
                self.count[p][d] = self.count[p].get(d, 0) + 1
        self.hist = [dict() for _ in range(n_phases)]
        for d, dest in enumerate(dests):
            for p in set(phases[d]) | ({dest.home} if dest.final else set()):
                self._add(self.hist[p], self._key(d, p, self.count[p].get(d, 0)), dest.weight)
        self.cost = [_hist_cost(h) for h in self.hist]

    def _key(self, d: int, p: int, n: int):
        dest = self.dests[d]
        fin = dest.final and p == dest.home
        return (n, fin) if (n or fin) else None

    @staticmethod
    def _add(hist: dict, key, k: int) -> None:
        if key is not None:
            hist[key] = hist.get(key, 0) + k
            if not hist[key]:
                del hist[key]

    def moved(self, d: int, p: int, n: int) -> dict:
        """Histogram of phase ``p`` with destination ``d`` contributing ``n`` there."""
        hist = dict(self.hist[p])
        w = self.dests[d].weight
        self._add(hist, self._key(d, p, self.count[p].get(d, 0)), -w)
        self._add(hist, self._key(d, p, n), w)
        return hist

    def apply(self, d: int, p: int, n: int, hist: dict, cost: int) -> None:
        self.hist[p], self.cost[p] = hist, cost
        if n:
            self.count[p][d] = n
        else:
            self.count[p].pop(d, None)


def total_cost(dests: list, phases: list, n_phases: int) -> int:
    return sum(_State(dests, phases, n_phases).cost)


def schedule(dests: list, n_phases: int, max_sweeps: int = 4, budget: int = 8000) -> tuple:
    """Deterministic local search from two starts, every contribution in its destination's home phase
    (today's schedule) and every contribution as early as it may run; the cheaper result wins, so no
    schedule is worse than the home one under the model.  ``budget`` bounds the phase evaluations of
    each start (compile time on the largest linkages).  Returns ``(phases per destination, cost of the
    home schedule, cost of the result)``."""
    home = [[d.home] * len(d.lo) for d in dests]
    before = total_cost(dests, home, n_phases)
    best = None
    for start in ([list(d.lo) for d in dests], home):
        phases, cost = _search(dests, n_phases, [list(p) for p in start], max_sweeps, budget)
        if best is None or cost < best[1]:
            best = (phases, cost)
    return best[0], before, best[1]


def _search(dests: list, n_phases: int, phases: list, max_sweeps: int, budget: int) -> tuple:
    """Moves: one contribution of a destination, or all of its contributions in one phase, to its
    earliest phase or to a phase the destination already visits; only strict improvements are
    accepted."""
    st = _State(dests, phases, n_phases)
    for _ in range(max_sweeps):
        improved = False
        for d, dest in enumerate(dests):
            moves = [([c], dest.lo[c]) for c in range(len(dest.lo))]
            for q in sorted(set(phases[d])):
                group = [c for c, x in enumerate(phases[d]) if x == q]
                if len(group) > 1:
                    moves.append((group, max(dest.lo[c] for c in group)))
            for group, lo in moves:
                ph = phases[d]
                for p in sorted({lo, dest.home} | {x for x in ph if x >= lo}):
                    if all(ph[c] == p for c in group):
                        continue
                    new = list(ph)
                    for c in group:
                        new[c] = p
                    touched = set(ph) | {p}
                    budget -= len(touched)
                    if budget < 0:
                        return phases, sum(st.cost)
                    trial = {}
                    for q in touched:
                        n = new.count(q)
                        hist = st.moved(d, q, n)
                        trial[q] = (n, hist, _hist_cost(hist))
                    if sum(t[2] - st.cost[q] for q, t in trial.items()) < 0:
                        for q, t in trial.items():
                            st.apply(d, q, *t)
                        phases[d] = ph = new
                        improved = True
        if not improved:
            break
    return phases, sum(st.cost)
