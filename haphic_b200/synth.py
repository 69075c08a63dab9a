"""Synthetic Hi-C inputs for tests and bench (SURVEY.md section 8(d)).

Nothing here is on the product path: it only fabricates inputs with the
shape the reference's own simulation tooling produces
(simulation/sim_contigs.py:43-104 names contigs
``{Chrom}_{n}_{start}_{end}_{ori}_{len}``), so that truth can be recovered
from contig names the way simulation/result_statistics.py does.

Model
-----
* ``nchr`` chromosomes of equal length; contigs are cut left to right with
  lengths ~ Normal(mean, 0.3*mean) truncated at >= ``min_len``; orientation is
  Bernoulli(0.5).
* read pairs: with probability ``cis_frac`` both ends fall on one chromosome,
  the first uniformly, the second at a genomic separation drawn from
  P(s) ~ 1/s on [1 kb, chrom_len] (reflected into the chromosome); otherwise
  both ends are uniform over the whole genome.
* a pair record is ``(ctg_a, pos_a, ctg_b, pos_b)`` int32, positions 0-based
  on the contig *as assembled* (i.e. reversed for '-' contigs) -- exactly the
  tuple the reference's generators yield (HapHiC_cluster.py:1562-1593) after
  name -> id translation.  Intra-contig pairs are left in the stream: dropping
  them (``ref != mref``, HapHiC_cluster.py:1582) is part of the path under test.
"""

from __future__ import annotations

import dataclasses
import math

import numpy as np
import torch


@dataclasses.dataclass
class Assembly:
    names: list            # contig names, FASTA order
    lengths: np.ndarray    # int64 [n]
    chrom: np.ndarray      # int32 [n] chromosome of each contig
    start: np.ndarray      # int64 [n] 0-based start of the contig on its chromosome
    ori: np.ndarray        # int8  [n] 1 = reverse-complemented
    chrom_len: int
    nchr: int

    @property
    def n(self) -> int:
        return len(self.names)


def make_assembly(nchr: int, n_contigs: int, mean_len: int, seed: int = 12345,
                  min_len: int = 5000, cv: float = 0.3, prefix: str = "Chr") -> Assembly:
    """Cut ``nchr`` equal chromosomes into ~``n_contigs`` contigs in total."""
    rng = np.random.default_rng(seed)
    per_chr = max(1, n_contigs // nchr)
    chrom_len = per_chr * mean_len
    names, lengths, chrom, start, ori = [], [], [], [], []
    for c in range(nchr):
        # draw lengths until the chromosome is covered, then fix the tail so the
        # chromosome holds exactly ``per_chr`` contigs (keeps n deterministic)
        draw = rng.normal(mean_len, cv * mean_len, size=per_chr * 3).astype(np.int64)
        draw = draw[draw >= min_len][:per_chr]
        assert len(draw) == per_chr, "not enough contig lengths drawn"
        scale = chrom_len / draw.sum()
        lens = np.maximum((draw * scale).astype(np.int64), min_len)
        lens[-1] += chrom_len - lens.sum()
        if lens[-1] < min_len:       # push the deficit into the longest contig
            k = int(np.argmax(lens[:-1]))
            lens[k] -= (min_len - lens[-1])
            lens[-1] = min_len
        assert lens.sum() == chrom_len and (lens > 0).all()
        p = 0
        oris = rng.integers(0, 2, size=per_chr)
        for k, (ln, o) in enumerate(zip(lens.tolist(), oris.tolist()), 1):
            names.append("{}{}_{}_{}_{}_{}_{}".format(prefix, c + 1, k, p + 1, p + ln, "-" if o else "+", ln))
            lengths.append(ln)
            chrom.append(c)
            start.append(p)
            ori.append(o)
            p += ln
    return Assembly(names, np.asarray(lengths, np.int64), np.asarray(chrom, np.int32),
                    np.asarray(start, np.int64), np.asarray(ori, np.int8), int(chrom_len), nchr)


def make_pairs_range(asm: Assembly, lo: int, hi: int, seed: int = 12345, cis_frac: float = 0.85,
                     device: str | torch.device = "cpu", block: int = 1 << 22) -> torch.Tensor:
    """Records [lo, hi) of the (conceptually infinite) pair stream of ``seed``.  The stream is generated in
    independently seeded blocks, so any slicing -- one GPU taking everything, or N ranks taking contiguous
    shards -- sees exactly the same records."""
    parts = []
    b0, b1 = lo // block, (hi + block - 1) // block
    for b in range(b0, b1):
        blk = make_pairs(asm, block, seed=seed * 1000003 + b, cis_frac=cis_frac, device=device, chunk=block)
        s, e = max(lo, b * block) - b * block, min(hi, (b + 1) * block) - b * block
        parts.append(blk[s:e])
    if not parts:
        return torch.empty((0, 4), dtype=torch.int32, device=torch.device(device))
    return torch.cat(parts) if len(parts) > 1 else parts[0].contiguous()


def make_pairs(asm: Assembly, n_pairs: int, seed: int = 12345, cis_frac: float = 0.85,
               device: str | torch.device = "cpu", chunk: int = 1 << 24, homolog=None) -> torch.Tensor:
    """Return an int32 tensor [n_pairs, 4] of (ctg_a, pos_a, ctg_b, pos_b).

    ``homolog=(ploidy, frac)`` treats every ``ploidy`` consecutive chromosomes as the haplotypes of one
    chromosome (as simulation/sim_haplotypes.py lays them out) and re-maps the second end of a fraction ``frac`` of
    the cis pairs to the SAME locus (+- 500 bp) of another haplotype -- the collinear "allelic" Hi-C links that
    remove_allelic_HiC_links (HapHiC_cluster.py:474-692) detects by their concordance ratio."""
    dev = torch.device(device)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    L = asm.chrom_len
    nchr = asm.nchr
    # contigs are laid out chromosome by chromosome: genome coordinate = chrom*L + pos
    gstart = torch.as_tensor(asm.chrom.astype(np.int64) * L + asm.start, device=dev)
    glen = torch.as_tensor(asm.lengths, device=dev)
    gori = torch.as_tensor(asm.ori.astype(np.int64), device=dev)
    out = torch.empty((n_pairs, 4), dtype=torch.int32, device=dev)
    log_ratio = math.log(L / 1000.0)

    def locate(gpos):
        idx = torch.searchsorted(gstart, gpos, right=True) - 1
        off = gpos - gstart[idx]
        ln = glen[idx]
        off = torch.where(gori[idx] == 1, ln - 1 - off, off)
        return idx.to(torch.int32), off.to(torch.int32)

    done = 0
    while done < n_pairs:
        m = min(chunk, n_pairs - done)
        u = torch.rand((m, 5 if homolog is None else 8), generator=g, device=dev, dtype=torch.float64)
        is_cis = u[:, 0] < cis_frac
        chrom_a = torch.clamp((u[:, 1] * nchr).long(), max=nchr - 1)
        pos_a = torch.clamp((u[:, 2] * L).long(), max=L - 1)
        # cis mate: separation ~ 1/s on [1e3, L], random direction, reflected into [0, L)
        sep = (1000.0 * torch.exp(u[:, 3] * log_ratio)).long()
        sign = torch.where(u[:, 4] < 0.5, -1, 1)
        pos_c = pos_a + sign * sep
        pos_c = torch.where(pos_c < 0, -pos_c, pos_c)
        pos_c = torch.where(pos_c >= L, 2 * (L - 1) - pos_c, pos_c)
        pos_c = torch.clamp(pos_c, 0, L - 1)
        # trans mate: uniform over the genome (re-using u[:,3], u[:,4] as fresh uniforms)
        chrom_t = torch.clamp((u[:, 3] * nchr).long(), max=nchr - 1)
        pos_t = torch.clamp((u[:, 4] * L).long(), max=L - 1)
        g_a = chrom_a * L + pos_a
        g_b = torch.where(is_cis, chrom_a * L + pos_c, chrom_t * L + pos_t)
        if homolog is not None:
            ploidy, frac = int(homolog[0]), float(homolog[1])
            switch = is_cis & (u[:, 5] < frac)
            hap = chrom_a % ploidy
            other = (hap + 1 + torch.clamp((u[:, 6] * (ploidy - 1)).long(), max=ploidy - 2)) % ploidy
            pos_h = torch.clamp(pos_a + ((u[:, 7] - 0.5) * 1000.0).long(), 0, L - 1)
            g_b = torch.where(switch, (chrom_a - hap + other) * L + pos_h, g_b)
        ia, pa = locate(g_a)
        ib, pb = locate(g_b)
        out[done:done + m, 0] = ia
        out[done:done + m, 1] = pa
        out[done:done + m, 2] = ib
        out[done:done + m, 3] = pb
        done += m
    return out


def random_sequence(length: int, rng: np.random.Generator) -> str:
    return "".join(np.array(list("ACGT"))[rng.integers(0, 4, size=length)])


def write_fasta(asm: Assembly, path: str, seed: int = 12345, width: int = 0) -> None:
    """i.i.d. uniform ACGT sequence per contig (GATC every ~256 bp)."""
    rng = np.random.default_rng(seed)
    alphabet = np.frombuffer(b"ACGT", dtype=np.uint8)
    with open(path, "w") as f:
        for name, ln in zip(asm.names, asm.lengths.tolist()):
            seq = alphabet[rng.integers(0, 4, size=ln)].tobytes().decode()
            f.write(">{}\n".format(name))
            if width:
                for i in range(0, ln, width):
                    f.write(seq[i:i + width] + "\n")
            else:
                f.write(seq + "\n")


def write_pairs(asm: Assembly, pairs: np.ndarray, path: str) -> None:
    """4DN .pairs text, 1-based positions, 7 columns (readID chr1 pos1 chr2 pos2 strand1 strand2)."""
    names = asm.names
    with open(path, "w") as f:
        f.write("## pairs format v1.0\n#columns: readID chr1 pos1 chr2 pos2 strand1 strand2\n")
        for r, (a, pa, b, pb) in enumerate(pairs.tolist()):
            f.write("r{}\t{}\t{}\t{}\t{}\t+\t-\n".format(r, names[a], pa + 1, names[b], pb + 1))


@dataclasses.dataclass
class Misjoined:
    asm: Assembly          # the misjoined assembly (chrom / start / ori of a joined contig are its first member's)
    pairs: np.ndarray      # int32 [P, 4] the records re-expressed on it
    junctions: dict        # name of a joined contig -> 0-based positions where one member ends and the next begins


def make_misjoined(asm: Assembly, pairs, frac: float = 0.01, seed: int = 12345, prefix: str = "Mis") -> Misjoined:
    """Join about ``frac * asm.n`` groups of 2 to 5 contigs, each from a different chromosome, end to end into chimeric
    contigs ``{prefix}{k}``, and re-express the records on the result.  A joined contig takes the place of its first
    member in FASTA order; the other contigs keep their names and order."""
    rng = np.random.default_rng(seed)
    pairs = np.asarray(pairs)
    by_chrom = [list(rng.permutation(np.nonzero(asm.chrom == c)[0])) for c in range(asm.nchr)]
    n_groups = max(1, int(round(frac * asm.n)))
    groups = []
    for _ in range(n_groups):
        size = int(rng.integers(2, 6))
        chroms = [c for c in rng.permutation(asm.nchr).tolist() if by_chrom[c]][:size]
        if len(chroms) < 2:
            break
        groups.append([int(by_chrom[c].pop()) for c in chroms])
    first_of = {g[0]: k for k, g in enumerate(groups)}
    member = {c: k for k, g in enumerate(groups) for c in g}
    names, lengths, chrom, start, ori = [], [], [], [], []
    new_id = np.empty(asm.n, np.int64)
    shift = np.zeros(asm.n, np.int64)
    junctions = {}
    for c in range(asm.n):
        if c in member and c not in first_of:
            continue
        i = len(names)
        if c in first_of:
            g = groups[first_of[c]]
            name = "{}{}".format(prefix, first_of[c] + 1)
            p, cuts = 0, []
            for m in g:
                new_id[m], shift[m] = i, p
                p += int(asm.lengths[m])
                cuts.append(p)
            junctions[name] = cuts[:-1]
            names.append(name)
            lengths.append(p)
        else:
            new_id[c] = i
            names.append(asm.names[c])
            lengths.append(int(asm.lengths[c]))
        chrom.append(int(asm.chrom[c]))
        start.append(int(asm.start[c]))
        ori.append(int(asm.ori[c]))
    out = pairs.astype(np.int64)
    for e in (0, 2):
        ok = (out[:, e] >= 0) & (out[:, e] < asm.n)
        c = out[ok, e]
        out[ok, e + 1] += shift[c]
        out[ok, e] = new_id[c]
    mis = Assembly(names, np.asarray(lengths, np.int64), np.asarray(chrom, np.int32), np.asarray(start, np.int64),
                   np.asarray(ori, np.int8), asm.chrom_len, asm.nchr)
    return Misjoined(mis, out.astype(np.int32), junctions)
