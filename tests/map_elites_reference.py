"""numpy restatement of MAP-Elites (map_elites, DESIGN.md section 4.12): the cell map, the claim and insertion, the selection
and the archive statistics.  float64 with each operation separately rounded, as the kernels compute them, so the kernels must
match it bit for bit.  The weights of an entering offspring come from the C twin's `materialize` (group 1, no head)."""
import numpy as np

STREAM_SELECT = 3
COMPACT_THREADS = 1024


class Spec:
    """A descriptor: dims, low, high, cells; width = high - low in float64, as the host computes it."""

    def __init__(self, dims, low, high, cells):
        self.dims = [int(d) for d in dims]
        self.low = np.array(low, dtype=np.float64)
        self.width = np.array(high, dtype=np.float64) - self.low
        self.cells = [int(c) for c in cells]
        self.n_cells = int(np.prod(self.cells))

    def ctype(self):
        from simple_es_b200.engine import map_spec
        return map_spec(self.dims, self.low, self.low + self.width, self.cells)


def cell_index(bc, spec):
    """[n] int64 cell of each behaviour row of bc [n, state_dim]; -1 where a descriptor coordinate is NaN."""
    bc = np.asarray(bc, dtype=np.float64)
    c = np.zeros(bc.shape[0], dtype=np.int64)
    bad = np.zeros(bc.shape[0], dtype=bool)
    with np.errstate(invalid="ignore", over="ignore"):
        for j, d in enumerate(spec.dims):
            x = bc[:, d]
            bad |= np.isnan(x)
            s = ((x - spec.low[j]) / spec.width[j]) * np.float64(spec.cells[j])
            hi = spec.cells[j] - 1
            k = np.where(s < 1.0, 0, np.where(s >= np.float64(hi), hi, np.floor(np.where(np.isfinite(s), s, 0.0)))).astype(np.int64)
            c = c * spec.cells[j] + k
    return np.where(bad, -1, c)


def empty(spec, state_dim, D):
    """An empty archive: F NaN, B NaN, born -1, W 0."""
    return {"F": np.full(spec.n_cells, np.nan), "B": np.full((spec.n_cells, state_dim), np.nan),
            "born": np.full((spec.n_cells, 2), -1, dtype=np.int32), "W": np.zeros((spec.n_cells, D), dtype=np.float32)}


def insert(archive, spec, order, fitness, bc, gen, weights_of):
    """Archive after generation gen's insertion (a new dict; the input is not modified).  weights_of(ids) -> [len(ids), D] f32
    (twin.materialize of the generation's parents).  Returns (archive, entered ids)."""
    a = {k: v.copy() for k, v in archive.items()}
    fitness = np.asarray(fitness, dtype=np.float64)
    cells = cell_index(bc, spec)
    cells[np.isnan(fitness)] = -1
    seen, entered = set(), []
    for r, i in enumerate(np.asarray(order)):
        c = int(cells[i])
        if c < 0 or c in seen:                # the candidate of a cell is its placed offspring of smallest rank
            continue
        seen.add(c)
        if np.isnan(a["F"][c]) or fitness[i] > a["F"][c]:
            a["F"][c] = fitness[i]
            a["B"][c] = bc[i]
            a["born"][c] = (gen, i)
            entered.append((c, int(i)))
    if entered:
        ids = np.array([i for _, i in entered], dtype=np.int32)
        a["W"][[c for c, _ in entered]] = weights_of(ids)
    return a, [i for _, i in entered]


def stats(F):
    """(n_occ, best cell or -1, its fitness or NaN, QD score) in k_map_compact's order: lane t sums the occupied cells
    c = t (mod 1024) in ascending c from +0.0, then a halving tree."""
    F = np.asarray(F, dtype=np.float64)
    occ = ~np.isnan(F)
    n_occ = int(occ.sum())
    if n_occ == 0:
        best, bf = -1, np.nan
    else:
        idx = np.flatnonzero(occ)
        best = int(idx[np.argmax(F[idx])])            # argmax returns the first (lowest-index) maximum
        bf = F[best]
    pad = -(-F.size // COMPACT_THREADS) * COMPACT_THREADS
    G = np.zeros(pad)
    G[:F.size] = np.where(occ, F, 0.0)
    O = np.zeros(pad, dtype=bool)
    O[:F.size] = occ
    G, O = G.reshape(-1, COMPACT_THREADS), O.reshape(-1, COMPACT_THREADS)
    lane = np.zeros(COMPACT_THREADS)
    for row in range(G.shape[0]):
        lane = np.where(O[row], lane + G[row], lane)
    h = COMPACT_THREADS // 2
    while h > 0:
        lane = lane[:h] + lane[h:2 * h]
        h //= 2
    return n_occ, best, bf, float(lane[0])


def select_cells(twin, F, P, gen, seed):
    """[P] int64: the archive cell parent row i is drawn from, or -1 while the archive is empty."""
    occ = np.flatnonzero(~np.isnan(np.asarray(F)))
    if occ.size == 0:
        return np.full(P, -1, dtype=np.int64)
    r = np.array([int(twin.philox([i, gen, 0, 0], [seed, STREAM_SELECT])[0]) for i in range(P)], dtype=np.uint64)
    return occ[((r * np.uint64(occ.size)) >> np.uint64(32)).astype(np.int64)]


def select(twin, archive, P, gen, seed, seed_row):
    """[P, D] f32 parent table of generation gen."""
    cells = select_cells(twin, archive["F"], P, gen, seed)
    if cells[0] < 0:
        return np.repeat(np.asarray(seed_row, dtype=np.float32)[None], P, axis=0)
    return archive["W"][cells]
