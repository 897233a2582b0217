"""Control logic of the sort kernels (madrona_b200/csrc/kernels_sort.cu), modelled on the CPU:
the decoupled look-back of a onesweep tile reads kLookWindow predecessors at a time and
consumes them in order (stop at the first unpublished one and retry from it, finish at the
first inclusive prefix): it must produce the same exclusive prefix as walking one
predecessor at a time, whatever the publication timing."""
import numpy as np

AGG, INC = 1, 2


def serial_lookback(read, tile):
    excl, look = 0, tile - 1
    while True:
        flag, val = read(look)
        if flag == 0:
            continue
        excl += val
        if flag == INC:
            return excl
        look -= 1


def windowed_lookback(read, tile, window=8):
    excl, look, done = 0, tile - 1, False
    while not done:
        v = [read(look - j) if look - j >= 0 else (0, 0) for j in range(window)]
        stop, consumed = False, 0
        for flag, val in v:
            if not stop:
                if flag == 0:
                    stop = True
                else:
                    excl += val
                    consumed += 1
                    if flag == INC:
                        done, stop = True, True
        look -= consumed
    return excl


def test_windowed_lookback_equals_serial_walk_under_any_publication_order():
    rng = np.random.default_rng(2)
    for _ in range(300):
        tile = int(rng.integers(1, 60))
        counts = rng.integers(0, 50, size=tile)
        incl = np.cumsum(counts)
        # predecessor p publishes AGGREGATE at time a[p] and INCLUSIVE at time b[p] >= a[p]; tile 0 is inclusive at once
        a = rng.integers(0, 40, size=tile)
        b = a + rng.integers(0, 40, size=tile)
        a[0] = b[0] = 0
        for walk in (serial_lookback, windowed_lookback):
            clock = [0]

            def read(p):
                clock[0] += 1                       # every poll advances time: pending entries appear eventually
                if clock[0] >= b[p]:
                    return INC, int(incl[p])
                if clock[0] >= a[p]:
                    return AGG, int(counts[p])
                return 0, 0
            assert walk(read, tile) == int(incl[tile - 1]), (walk.__name__, tile)

