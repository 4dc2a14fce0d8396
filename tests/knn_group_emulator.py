"""A NumPy/float32 emulation of the GROUP PATH of csrc/gsx_sor.cu's query kernel (GSX_KNN_GROUP; test infrastructure).

A batch of `batch` consecutive sorted positions that share one grid cell and lie inside the centre probe's long bucket
(A) runs every member's seed-chunk scan, (B) walks the probes / supers / chunks ONCE with the box-to-box bound of the
batch's bounding box against tau_G = the largest seed tau, into a list of at most `group_list` chunk entries plus a set
of small buckets, and (C) per query tests only the listed chunks, then the listed small buckets, nearest box first with
its own bound.  A seed list that is not full or an overflowing list sends the batch to the per-query path, which is
tests/knn_emulator.py's `emulate` unchanged.  The kernel also requires the batch to lie in one 32-point chunk; here
each query keeps its own seed chunk, which covers that case.  Every float operation is a float32 NumPy scalar op in
the kernel's order, so the result must equal the brute-force oracle bit for bit.
"""
import numpy as np

from knn_emulator import D2LIM, P1, P2, P3, _d2, _lb, _probe_hash, emulate, f32


def _lb_box(blo, bhi, lo, hi):
    """Group bound: lower bound of _lb(q, lo, hi) for every q in the box [blo, bhi] (same op sequence)."""
    d = [max(max(f32(lo[a] - bhi[a]), f32(blo[a] - hi[a])), f32(0)) for a in range(3)]
    return f32(f32(f32(d[0] * d[0]) + f32(d[1] * d[1])) + f32(d[2] * d[2]))


def _grid(pos, chunk, fan, morton_bits):
    """The hash-sorted order, bucket ranges and boxes exactly as knn_emulator.emulate builds them."""
    n = len(pos)
    lo = pos.min(0)
    ext = pos.max(0) - lo
    vol = np.prod(ext)
    if vol <= 0:
        vol = 1.0
    avg = max(1e-8, vol / n)
    cell = f32(max(float((avg * 32) ** (1.0 / 3.0)), 1e-4))
    fr = (pos - lo) / cell
    gi = np.floor(fr).astype(np.int32).astype(np.int64)
    h = ((gi[:, 0] * P1) ^ (gi[:, 1] * P2) ^ (gi[:, 2] * P3)) % n
    sub = np.minimum((fr - np.floor(fr)) * (1 << morton_bits), (1 << morton_bits) - 1).astype(np.int64)
    mort = np.zeros(n, np.int64)
    for b in range(morton_bits):
        for a in range(3):
            mort |= ((sub[:, a] >> b) & 1) << (3 * b + (2 - a))
    order = np.lexsort((np.arange(n), mort, h))
    sp = pos[order]
    start, end = {}, {}
    for j, hv in enumerate(h[order]):
        start.setdefault(int(hv), j)
        end[int(hv)] = j + 1
    box = {hv: (sp[start[hv]:end[hv]].min(0), sp[start[hv]:end[hv]].max(0)) for hv in start}
    nchunk = (n + chunk - 1) // chunk
    cbox = [(sp[c * chunk:(c + 1) * chunk].min(0), sp[c * chunk:(c + 1) * chunk].max(0)) for c in range(nchunk)]
    sup = chunk * fan
    sbox = [(sp[s * sup:(s + 1) * sup].min(0), sp[s * sup:(s + 1) * sup].max(0)) for s in range((n + sup - 1) // sup)]
    cells = np.floor((sp - lo) / cell).astype(np.int32)
    return order, sp, cells, start, end, box, cbox, sbox


def emulate_group(pos, k, mode="i32wrap", chunk=4, fan=4, small_bucket=6, morton_bits=2, flat_supers=0, group=32,
                  batch=4, group_list=64):
    """final_means float32[N] with the group path on (batch > 0, K <= 32), and counters {group_queries,
    group_fallbacks}.  The other parameters are those of knn_emulator.emulate."""
    pos = np.ascontiguousarray(pos, dtype=np.float32)
    out, _ = emulate(pos, k, mode, chunk=chunk, fan=fan, small_bucket=small_bucket, morton_bits=morton_bits,
                     flat_supers=flat_supers, group=group)          # the per-query path of every query
    n = len(pos)
    K = min(k, 50)
    stats = dict(group_queries=0, group_fallbacks=0)
    if K > 32:
        return out, stats
    order, sp, cells, start, end, box, cbox, sbox = _grid(pos, chunk, fan, morton_bits)

    def probes_of(g):
        return [hv if hv in start else None for hv in
                (_probe_hash(int(g[0]) + dx, int(g[1]) + dy, int(g[2]) + dz, n, mode)
                 for dx in (-1, 0, 1) for dy in (-1, 0, 1) for dz in (-1, 0, 1))]

    def scan(q, lst, j0, j1):                               # visit candidates [j0, j1) into the ascending list
        for j in range(j0, j1):
            d2 = _d2(q, sp[j])
            if d2 > f32(1.0e-12) and d2 < lst[K - 1]:
                lst = sorted(lst + [d2])[:K]
        return lst

    for b0 in range(0, n, batch):
        b1 = min(b0 + batch, n)
        if any((cells[t] != cells[b0]).any() for t in range(b0, b1)):
            continue
        probes = probes_of(cells[b0])
        h13 = probes[13]
        if h13 is None or end[h13] - start[h13] <= small_bucket or not (start[h13] <= b0 and b1 <= end[h13]):
            continue
        # phase A: the seed chunk of every member
        seeds = []
        for t in range(b0, b1):
            c = t // chunk
            seeds.append(scan(sp[t], [D2LIM] * K, max(c * chunk, start[h13]), min((c + 1) * chunk, end[h13])))
        if any(not (s_[K - 1] < D2LIM) for s_ in seeds):
            stats["group_fallbacks"] += 1
            continue
        # phase B: one walk for the batch, probe multiplicity kept
        tau_g = max(s_[K - 1] for s_ in seeds)
        blo, bhi = sp[b0:b1].min(0), sp[b0:b1].max(0)
        entries, small = [], []
        for p, hv in enumerate(probes):
            if hv is None or not (_lb_box(blo, bhi, *box[hv]) < tau_g):
                continue
            s, e = start[hv], end[hv]
            if e - s <= small_bucket:
                small.append(p)
                continue
            fc, lc = s // chunk, (e - 1) // chunk
            if flat_supers > 0 and lc // fan - fc // fan < flat_supers:
                cands = range(fc, lc + 1)
            else:
                cands = [c for sid in range(fc // fan, lc // fan + 1) if _lb_box(blo, bhi, *sbox[sid]) < tau_g
                         for c in range(sid * fan, sid * fan + fan) if fc <= c <= lc]
            entries += [(c, p) for c in cands if _lb_box(blo, bhi, *cbox[c]) < tau_g]
        if len(entries) > group_list:
            stats["group_fallbacks"] += 1
            continue
        # phase C: per query, the listed chunks 32 at a time, then the small buckets, nearest box first
        for t in range(b0, b1):
            stats["group_queries"] += 1
            q, lst = sp[t], list(seeds[t - b0])
            own = (t // chunk, 13)                          # the seed chunk, already scanned
            for g0 in range(0, len(entries), 32):
                keyed = [(_lb(q, *cbox[c]), e0, c, p) for e0, (c, p) in enumerate(entries[g0:g0 + 32])
                         if (c, p) != own]
                keyed = [x for x in keyed if x[0] < lst[K - 1]]
                while keyed:
                    x = min(keyed)                          # nearest box first, lowest list index on ties
                    if not (x[0] < lst[K - 1]):
                        break
                    keyed.remove(x)
                    hv = probes[x[3]]
                    lst = scan(q, lst, max(x[2] * chunk, start[hv]), min((x[2] + 1) * chunk, end[hv]))
            pk = {p: _lb(q, *box[probes[p]]) for p in small}
            while pk:
                p = min(pk, key=lambda u: (pk[u], u))
                if not (pk[p] < lst[K - 1]):
                    break
                del pk[p]
                lst = scan(q, lst, start[probes[p]], end[probes[p]])
            vals = [v for v in (np.sqrt(v) for v in lst) if v < f32(0.9e10)]
            ssum = f32(0)
            for v in vals:
                ssum = f32(ssum + v)
            out[order[t]] = f32(ssum / f32(len(vals))) if vals else f32(0)
    return out, stats
