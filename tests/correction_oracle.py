"""numpy restatement of the reference's assembly correction (scripts/HapHiC_cluster.py v1.0.7: parse_pairs_for_correction
1300-1344, detect_break_points 943-1014, break_and_update_ctgs / correct_assembly 1017-1297, convert_ctg 1405-1411) for the
tests.  It keeps the reference's data model -- one int32 numpy array per contig, fragments as views of their parent, the
links of every ctg_link_pos_dict key, pos_shift's keys -- with the per-pair loops vectorised so that it follows at
200M pairs."""

import numpy as np


def pass1(rec, lengths, res):
    """Coverage (concatenated per contig, len // res + 1 bins each), bin offsets and the same-contig links (ctg, lo, hi)."""
    rec = np.asarray(rec)
    lengths = np.asarray(lengths, np.int64)
    n = len(lengths)
    m = (rec[:, 0] == rec[:, 2]) & (rec[:, 0] >= 0) & (rec[:, 0] < n)
    c = rec[m, 0].astype(np.int64)
    lo = np.minimum(rec[m, 1], rec[m, 3]).astype(np.int64)
    hi = np.maximum(rec[m, 1], rec[m, 3]).astype(np.int64)
    off = np.concatenate([[0], np.cumsum(lengths // res + 1)])
    nb = int(off[-1])
    diff = np.bincount(off[c] + lo // res, minlength=nb + 1) - np.bincount(off[c] + hi // res + 1, minlength=nb + 1)
    cov = np.cumsum(diff[:nb]).astype(np.int32)
    return cov, off, c, lo, hi


def detect_one(cov, length, res, median_cov_ratio, region_len_ratio, min_region_cutoff):
    """detect_break_points for one fragment: [(breakpoint, coverage), ...] or None."""
    median_cov = np.median(cov)
    if not median_cov:
        return None
    cov_cutoff = median_cov * median_cov_ratio
    high = (cov >= cov_cutoff).astype(np.int8)
    d = np.diff(np.concatenate([[0], high, [0]]))
    starts, ends = np.nonzero(d == 1)[0].tolist(), np.nonzero(d == -1)[0].tolist()
    if len(starts) < 2:
        return None
    region_cutoff = max(min_region_cutoff, length * region_len_ratio)
    kept = [(s, e) for s, e in zip(starts, ends) if (e - s) * res >= region_cutoff]
    if len(kept) < 2:
        return None
    cands, any_zero = [], False
    for (_s0, e0), (s1, _e1) in zip(kept[:-1], kept[1:]):
        v = cov[e0:s1]
        z = np.nonzero(v == 0)[0]
        if len(z):
            any_zero = True
            cands.append((int(z[0]) + e0, 0))
        else:
            a = int(v.argmin())
            cands.append((a + e0, int(v[a])))
    if any_zero:
        return [(b * res, 0) for b, cv in cands if cv == 0]
    b, cv = sorted(cands, key=lambda x: x[1])[0]
    return [(b * res, cv)]


def _pos_shift_key(ctg, n, shift, length, unbroken):
    if ctg in unbroken:
        start, end = 1, length
    else:
        ctg, rng = ctg.rsplit(":", 1)
        start, end = [int(p) for p in rng.split("-")]
    p = shift[n]
    return "{}:{}-{}".format(ctg, p + start, shift[n - 1] if n else end)


def correct(rec, names, lengths, res, nrounds, median_cov_ratio=0.2, region_len_ratio=0.1, min_region_cutoff=5000):
    """correct_assembly without sequences.  Returns a dict with the per-round breakpoint dicts, the final dicts, the
    corrected fa_dict order (names, lengths) and the pass-1 arrays."""
    cov, off, c, lo, hi = pass1(rec, lengths, res)
    cov_all = cov.copy()
    fa = {n: int(L) for n, L in zip(names, np.asarray(lengths).tolist())}
    ctg_cov = {n: cov_all[off[i]:off[i + 1]] for i, n in enumerate(names)}          # views, as the reference slices
    order = np.argsort(c, kind="stable")
    cuts = np.searchsorted(c[order], np.arange(len(names) + 1))
    links = {names[i]: [(lo[order[cuts[i]:cuts[i + 1]]], hi[order[cuts[i]:cuts[i + 1]]])]
             for i in range(len(names)) if cuts[i + 1] > cuts[i]}
    unbroken = set(names)
    src, fpos, ffrag = {}, {}, {}
    rounds = []
    nbroken = 0
    for nround in range(nrounds):
        bpd = {}
        for ctg, cl in ctg_cov.items():
            r = detect_one(cl, fa[ctg], res, median_cov_ratio, region_len_ratio, min_region_cutoff)
            if r:
                bpd[ctg] = r
        rounds.append(bpd)
        if nround == 0:
            nbroken = len(bpd)
        if not bpd:
            break
        if nround == 0:
            for ctg in bpd:
                src[ctg], fpos[ctg], ffrag[ctg] = ctg, [0], [ctg]
        last = nround + 1 == nrounds
        before = set(fa)
        for ctg, bps in bpd.items():
            if not last:
                shift = [p for p, _ in bps][::-1] + [0]
                parts = links.get(ctg, [])
                L = np.concatenate([p[0] for p in parts]) if parts else np.zeros(0, np.int64)
                H = np.concatenate([p[1] for p in parts]) if parts else np.zeros(0, np.int64)
                if bps[0][1] != 0:
                    bp = bps[0][0]
                    span = (L <= bp + res) & (H >= bp)
                    view = ctg_cov[ctg]
                    d = (np.bincount(L[span] // res, minlength=len(view) + 1) -
                         np.bincount(H[span] // res + 1, minlength=len(view) + 1))
                    view -= np.cumsum(d)[:len(view)].astype(np.int32)
                    L, H = L[~span], H[~span]
                asc = np.array(shift[::-1], np.int64)
                ni = len(shift) - np.searchsorted(asc, L, side="right")
                nj = len(shift) - np.searchsorted(asc, H, side="right")
                same = ni == nj
                for n in np.unique(ni[same]).tolist():
                    sel = same & (ni == n)
                    key = _pos_shift_key(ctg, n, shift, fa[ctg], unbroken)
                    links.setdefault(key, []).append((L[sel] - shift[n], H[sel] - shift[n]))
            start = 0
            s0 = src[ctg]
            fi = ffrag[s0].index(ctg)
            fp = fpos[s0][fi]
            ffrag[s0].pop(fi)
            fpos[s0].pop(fi)
            if ctg not in unbroken:
                raw, rng = ctg.rsplit(":", 1)
                sh = int(rng.split("-")[0]) - 1
            else:
                raw, sh = ctg, 0
            last_point = 0
            pieces = []
            for n, (point, _) in enumerate(bps, 1):
                s = 1 if n == 1 else last_point + 1
                last_point = point
                pieces.append(("{}:{}-{}".format(raw, s + sh, point + sh), start, point))
                start = point
            pieces.append(("{}:{}-{}".format(raw, sh + last_point + 1, sh + fa[ctg]), start, fa[ctg]))
            for k, (new, a, b) in enumerate(pieces):
                src[new] = s0
                ffrag[s0].insert(fi, new)
                fpos[s0].insert(fi, fp + a)
                if not last:
                    ctg_cov[new] = ctg_cov[ctg][a // res:b // res] if k + 1 < len(pieces) else ctg_cov[ctg][a // res:]
                fa[new] = b - a
            del fa[ctg]
            if not last:
                del ctg_cov[ctg]
        if not last:
            for ctg in before - set(bpd):
                ctg_cov.pop(ctg, None)
        unbroken -= set(bpd)
    return dict(rounds=rounds, nbroken=nbroken, final_pos=fpos, final_frag=ffrag, names=list(fa), lengths=list(fa.values()),
                cov=cov, bin_off=off, link_ctg=c, link_lo=lo, link_hi=hi)


def remap(rec, names, result):
    """The second pass's records: every end on a broken contig moves to its piece (largest start <= pos), ids follow the
    corrected fa_dict order; ids outside the FASTA stay -1."""
    new_id = {n: i for i, n in enumerate(result["names"])}
    key, ids, starts = [], [], []
    for i, n in enumerate(names):
        if n in result["final_frag"]:
            st = result["final_pos"][n][::-1]
            fr = result["final_frag"][n][::-1]
        else:
            st, fr = [0], [n]
        key += [(i << 32) + s for s in st]
        starts += st
        ids += [new_id[f] for f in fr]
    key, ids, starts = np.array(key, np.int64), np.array(ids, np.int64), np.array(starts, np.int64)
    out = np.asarray(rec).astype(np.int64).copy()
    for e in (0, 2):
        c, pos = out[:, e], out[:, e + 1]
        bad = (c < 0) | (c >= len(names))
        k = np.searchsorted(key, (np.where(bad, 0, c) << 32) + pos, side="right") - 1
        out[:, e] = np.where(bad, -1, ids[k])
        out[:, e + 1] = np.where(bad, pos, pos - starts[k])
    return out.astype(np.int32)
