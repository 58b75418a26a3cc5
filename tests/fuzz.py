"""Random adversarial bundles built directly in the agpu_batch_in layout (no synthetic transcriptome behind them): ragged
CIGARs with every op the reference walks (M I D N S = X), heavy position ties, qname groups of 1-4 hits with consistent or
inconsistent mate fields, empty bundles.  Used by the CPU tier (kernel-logic build) and the -m gpu tier alike."""
import numpy as np

from aletsch_b200 import hostlib as H

M, I, D, N, S, EQ, X = 0, 1, 2, 3, 4, 7, 8
REF_OPS = (M, D, N, EQ, X)


def random_cigar(rng, spliced):
    ops = []
    if rng.random() < 0.15:
        ops.append((S, int(rng.integers(1, 12))))
    nblocks = int(rng.integers(1, 5)) if spliced else int(rng.integers(1, 3))
    for k in range(nblocks):
        kind = M if rng.random() < 0.93 else (EQ if rng.random() < 0.5 else X)
        ops.append((kind, int(rng.integers(1, 70))))
        if k + 1 < nblocks:
            r = rng.random()
            if spliced and r < 0.7:
                ops.append((N, int(rng.integers(20, 400))))
            elif r < 0.85:
                ops.append((D, int(rng.integers(1, 6))))
            else:
                ops.append((I, int(rng.integers(1, 6))))
    if rng.random() < 0.15:
        ops.append((S, int(rng.integers(1, 12))))
    return ops


def random_bundle(rng, n_hits, strand, exon_grid, pair_heavy=False):
    """hits sorted by pos with no neighbour equal in (pos, rpos); splice positions are drawn from a small grid so that chains,
    junctions and coverage borders collide a lot"""
    pos = np.sort(rng.integers(1000, 1000 + (3 if pair_heavy else 40) * max(n_hits, 1) + 200, n_hits)).astype(np.int32)
    cig, cig_off, rpos = [], [0], []
    for i in range(n_hits):
        spliced = rng.random() < 0.45
        ops = random_cigar(rng, spliced)
        if spliced and exon_grid:
            # snap block lengths so that splice sites fall on a coarse grid (shared junctions)
            ops = [(o, (l // 8 + 1) * 8 if o in (M, N) else l) for o, l in ops]
            pos[i] = (pos[i] // 8) * 8
        p = int(pos[i])
        for o, l in ops:
            if o in REF_OPS:
                p += l
            cig.append((l << 4) | o)
        cig_off.append(len(cig))
        rpos.append(p)
    pos = np.maximum.accumulate(pos)            # snapping may have broken the order
    rpos = np.array([r - int(p0) + int(p1) for r, p0, p1 in zip(rpos, pos, pos)], np.int32) if n_hits else np.zeros(0, np.int32)
    # recompute rpos from the final pos
    rp = []
    for i in range(n_hits):
        p = int(pos[i])
        for c in cig[cig_off[i]:cig_off[i + 1]]:
            if (c & 0xF) in REF_OPS:
                p += c >> 4
        rp.append(p)
    rpos = np.array(rp, np.int32) if n_hits else np.zeros(0, np.int32)
    # the packing contract: no hit equals its predecessor in (pos, rpos) -> drop such hits
    keep = [i for i in range(n_hits) if i == 0 or not (pos[i] == pos[i - 1] and rpos[i] == rpos[i - 1])]
    # keep must be re-checked against the previous KEPT hit
    kept = []
    for i in keep:
        if kept and pos[i] == pos[kept[-1]] and rpos[i] == rpos[kept[-1]]:
            continue
        kept.append(i)
    n = len(kept)
    out = {"pos": pos[kept], "rpos": rpos[kept]}
    cg, co = [], [0]
    for i in kept:
        cg.extend(cig[cig_off[i]:cig_off[i + 1]])
        co.append(len(cg))
    out["cigar"] = np.array(cg, np.uint32)
    out["cigar_off"] = np.array(co, np.uint32)
    # mates: qname groups of size 1-4
    qid = np.zeros(n, np.uint64)
    mpos = rng.integers(900, 3000, n).astype(np.int32)
    isize = rng.integers(-400, 400, n).astype(np.int32)
    perm = rng.permutation(n)
    k = 0
    q = 1
    while k < n:
        g = int(min(n - k, rng.choice([1, 2, 2, 2, 2, 3, 4])))
        members = np.sort(perm[k:k + g])
        qid[members] = q + int(rng.integers(0, 1 << 40)) * 4096
        if g >= 2:
            a, b = int(members[0]), int(members[-1])
            mpos[a] = out["pos"][b]
            mpos[b] = out["pos"][a]
            sz = int(rng.integers(50, 500))
            isize[a], isize[b] = sz, -sz
            if rng.random() < 0.1:
                isize[b] += 1                      # inconsistent pair: must stay unpaired
            for m in members[1:-1]:                # extra alignments of the same read compete for the mate
                mpos[int(m)] = out["pos"][b]
                isize[int(m)] = sz if rng.random() < 0.5 else int(rng.integers(1, 500))
        q += 1
        k += g
    if pair_heavy and n:
        # candidate relations that are anything but isolated pairs: query names shared by up to 8 hits, mpos pointing at the
        # position of a random member of the same group (possibly the hit's own), isize from a handful of values incl. 0
        perm = rng.permutation(n)
        k = 0
        while k < n:
            g = int(min(n - k, rng.choice([1, 2, 2, 3, 4, 5, 8])))
            members = perm[k:k + g]
            name = np.uint64(int(rng.integers(1, 1 << 50)))
            for x in members:
                qid[int(x)] = name
                mpos[int(x)] = out["pos"][int(rng.choice(members))]
                isize[int(x)] = int(rng.choice([-60, -50, 0, 50, 60, 50, -50]))
            k += g
    out["qid"] = qid
    out["mpos"] = mpos
    out["isize"] = isize
    out["flag"] = rng.integers(0, 4096, n).astype(np.uint16)
    out["strand"] = np.full(n, ord(strand), np.uint8)
    xs = np.full(n, ord("."), np.uint8)
    for j in range(n):
        has_n = any((c & 0xF) == N for c in out["cigar"][out["cigar_off"][j]:out["cigar_off"][j + 1]])
        if has_n:
            xs[j] = ord(strand) if (strand != "." and rng.random() < 0.9) else ord(rng.choice(["+", "-"]))
    out["xs"] = xs
    return out


def random_batch(seed, n_bundles=12, max_hits=60, empty_every=0, exon_grid=True, pair_heavy=False):
    rng = np.random.default_rng(seed)
    parts = []
    for k in range(n_bundles):
        if empty_every and k % empty_every == empty_every - 1:
            n = 0
        else:
            n = int(rng.integers(1, max_hits + 1))
        parts.append(random_bundle(rng, n, str(rng.choice(["+", "-"])), exon_grid, pair_heavy))
    arr = {f: (np.concatenate([p[f] for p in parts]).astype(dt) if parts else np.zeros(0, dt)) for f, dt in H.HIT_FIELDS}
    hit_off = np.zeros(len(parts) + 1, np.int64)
    cig_off = [np.zeros(1, np.uint32)]
    cbase = 0
    for i, p in enumerate(parts):
        hit_off[i + 1] = hit_off[i] + len(p["pos"])
        cig_off.append(p["cigar_off"][1:] + np.uint32(cbase))
        cbase += len(p["cigar"])
    arr["bundle_hit_off"] = hit_off
    arr["cigar_off"] = np.concatenate(cig_off).astype(np.uint32)
    arr["cigar"] = np.concatenate([p["cigar"] for p in parts]).astype(np.uint32) if parts else np.zeros(0, np.uint32)
    arr["bundle_tid"] = np.zeros(len(parts), np.int32)
    arr["bundle_sample"] = np.zeros(len(parts), np.int32)
    arr["bundle_side"] = np.zeros(len(parts), np.uint8)
    return H.PackedBatch(arr)


def strand_clusters(batch, rng):
    """random clusters of 2-5 bundles of one strand (assembler::bridge asserts equal strands, meta/bundle.cc:93)"""
    a = batch.a
    off = a["bundle_hit_off"]
    st = [int(a["strand"][int(off[k])]) if off[k + 1] > off[k] else -1 for k in range(batch.n_bundles)]      # -1: empty bundle, left out
    groups = []
    for s in sorted(set(st) - {-1}):
        ks = [k for k in range(batch.n_bundles) if st[k] == s]
        rng.shuffle(ks)
        while len(ks) >= 2:
            n = min(len(ks), int(rng.integers(2, 5)))
            if len(ks) - n == 1:
                n += 1
            groups.append([int(x) for x in ks[:n]])
            ks = ks[n:]
    return groups


def dag_bundle(n_exons, reads_per_junction=1, strand="+", pairs=3, exon_len=20, step=100, base=1000):
    """one bundle whose splice graph is a complete DAG: n_exons exons of exon_len bases, a junction from every exon to every
    later one (reads_per_junction + (i + j) % 3 spliced reads each, so the weights differ), and `pairs` read pairs with one
    mate in the first exon and the other in the last.  Every pair is one cluster whose bridging range holds all exons, so the
    bridging DP of the last exons sees up to K candidates from each earlier exon."""
    X = [base + step * i for i in range(n_exons)]
    hits = []        # (pos, cigar ops, qid, mpos, isize, flag)
    q = 1
    for i in range(n_exons):
        for j in range(i + 1, n_exons):
            for r in range(reads_per_junction + (i + j) % 3):
                a = exon_len // 2 + r % (exon_len // 2 - 1)       # the read starts a bases into exon i
                p = X[i] + a
                ops = [(M, exon_len - a), (N, X[j] - X[i] - exon_len), (M, 3 + r % 5)]
                hits.append((p, ops, q, 0, 0, 0))
                q += 1
    for k in range(pairs):
        p1, p2 = X[0] + k, X[-1] + 1 + k
        sz = p2 + 12 - p1
        hits.append((p1, [(M, 12)], q, p2, sz, 0x1 | 0x2 | 0x20 | 0x40))
        hits.append((p2, [(M, 12)], q, p1, -sz, 0x1 | 0x2 | 0x10 | 0x80))
        q += 1
    hits.sort(key=lambda h: (h[0], sum(l for o, l in h[1] if o in REF_OPS)))
    out = {"pos": np.array([h[0] for h in hits], np.int32)}
    cig, co, rp = [], [0], []
    for h in hits:
        cig.extend((l << 4) | o for o, l in h[1])
        co.append(len(cig))
        rp.append(h[0] + sum(l for o, l in h[1] if o in REF_OPS))
    out["rpos"] = np.array(rp, np.int32)
    out["cigar"] = np.array(cig, np.uint32)
    out["cigar_off"] = np.array(co, np.uint32)
    out["qid"] = np.array([h[2] for h in hits], np.uint64)
    out["mpos"] = np.array([h[3] for h in hits], np.int32)
    out["isize"] = np.array([h[4] for h in hits], np.int32)
    out["flag"] = np.array([h[5] for h in hits], np.uint16)
    out["strand"] = np.full(len(hits), ord(strand), np.uint8)
    out["xs"] = np.array([ord(strand) if len(h[1]) > 1 else ord(".") for h in hits], np.uint8)
    return out


def pack_bundles(parts):
    """a PackedBatch of bundles given as dicts of hit arrays (as random_bundle returns them)"""
    arr = {f: (np.concatenate([p[f] for p in parts]).astype(dt) if parts else np.zeros(0, dt)) for f, dt in H.HIT_FIELDS}
    hit_off = np.zeros(len(parts) + 1, np.int64)
    cig_off = [np.zeros(1, np.uint32)]
    cbase = 0
    for i, p in enumerate(parts):
        hit_off[i + 1] = hit_off[i] + len(p["pos"])
        cig_off.append(p["cigar_off"][1:] + np.uint32(cbase))
        cbase += len(p["cigar"])
    arr["bundle_hit_off"] = hit_off
    arr["cigar_off"] = np.concatenate(cig_off).astype(np.uint32)
    arr["cigar"] = np.concatenate([p["cigar"] for p in parts]).astype(np.uint32) if parts else np.zeros(0, np.uint32)
    arr["bundle_tid"] = np.zeros(len(parts), np.int32)
    arr["bundle_sample"] = np.zeros(len(parts), np.int32)
    arr["bundle_side"] = np.zeros(len(parts), np.uint8)
    return H.PackedBatch(arr)
