"""The bookkeeping of a shared pass (internal.h LapState, DESIGN.md section 4 "two searches in flight"), restated in
Python: a lap claims the chunks of its segments front to back and seals a segment at its first claim; a joiner
atomicCAS-es every segment word that is still 0 and catches up, in a lap of its own, over the segments it did not get;
that catch-up can be joined in turn.  For every interleaving of claims and joins, every segment is scanned exactly
once per query, so `covered` equals the table's rows for each of them."""
import itertools

SEGS = 6            # small enough to try every join point
SEALED, JOINED = 1 << 31, 1


class Lap:
    """one lap: its segment words and the segments it scans, in claim order"""

    def __init__(self, segs):
        self.word = [0 if s in segs else SEALED for s in range(SEGS)]   # outside the list: closed to joiners
        self.todo = list(segs)
        self.scanned = {}                                              # segment -> queries that scored it

    def claim(self):
        s = self.todo.pop(0)
        old = self.word[s]
        self.word[s] |= SEALED                                         # atomicOr: the same set for every claimer
        self.scanned[s] = ["primary"] + (["joiner"] if old & JOINED else [])


def join(host):
    """the join kernel: the segments got, and the joiner's own lap over the others"""
    got = []
    for s in range(SEGS):
        if host.word[s] == 0:                                          # atomicCAS(0 -> JOINED)
            host.word[s] = JOINED
            got.append(s)
    return got, Lap([s for s in range(SEGS) if s not in got])


def coverage(lap_a, got, lap_b):
    a = sorted(lap_a.scanned)
    b = sorted([s for s in got if "joiner" in lap_a.scanned.get(s, [])] + list(lap_b.scanned))
    return a, b


def test_every_join_point_covers_each_segment_once_per_query():
    for t in range(SEGS + 1):                                          # the join lands after t claims of the lap
        a = Lap(range(SEGS))
        for _ in range(t):
            a.claim()
        got, b = join(a)
        assert got == list(range(t, SEGS))
        while a.todo:
            a.claim()
        while b.todo:                                                  # the catch-up runs after the lap (event wait)
            b.claim()
        ca, cb = coverage(a, got, b)
        assert ca == list(range(SEGS)) and cb == list(range(SEGS)), t


def test_a_catch_up_is_joinable_and_its_joiner_still_covers_everything():
    for t, u in itertools.product(range(SEGS + 1), range(SEGS + 1)):
        a = Lap(range(SEGS))
        for _ in range(t):
            a.claim()
        got_b, b = join(a)
        while a.todo:
            a.claim()
        for _ in range(min(u, len(b.todo))):
            b.claim()
        got_c, c = join(b)                                             # the third search joins the catch-up
        assert not set(got_c) & set(got_b)                             # the segments b got in a stay closed to c
        while b.todo:
            b.claim()
        while c.todo:
            c.claim()
        cov_c = sorted([s for s in got_c if "joiner" in b.scanned.get(s, [])] + list(c.scanned))
        assert cov_c == list(range(SEGS)), (t, u)
        _, cov_b = coverage(a, got_b, b)
        assert cov_b == list(range(SEGS)), (t, u)


def test_a_join_after_the_last_seal_is_a_full_catch_up():
    a = Lap(range(SEGS))
    while a.todo:
        a.claim()
    got, b = join(a)
    assert got == [] and b.todo == list(range(SEGS))
