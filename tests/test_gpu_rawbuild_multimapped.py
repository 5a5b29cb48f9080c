"""Device class assignment for multimapped samples (sbq_set_raw_mass_mode(SBQ_RAW_MASS_ANY)): fragment masses are 1/NH
fractions, so the float class mass n_c = (int) sum (float)mass over ExonBin::_frags (include/isoform.h:285-296) depends on the
order of the sum, which is std::set<Contig> order (ref_id, then the feature lists lexicographically by (offset, len), op codes
ignored, a proper prefix first). The CPU test restates that sum in Python and checks the host builder (and the compiled
reference, where it is built) against it on inputs where a wrong order gives other bits; the GPU tests check the device tables in
ANY mode against the host builder, bit for bit."""
import os

import numpy as np
import pytest

import locusgen
from test_builder import reference_table, specs_for

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIG = 12345.678


def fractional(hits, seed):
    """(mass, ...) tuples with every mass m replaced by m / NH (NH seeded from 2..8); about one hit in 25 also carries a large
    member (BIG), so that the float sum of a class depends on where in the order that member comes."""
    rng = np.random.default_rng(seed + 991)
    nh = rng.integers(2, 9, len(hits))
    big = rng.random(len(hits)) < 0.04
    return [((BIG if b else 0.0) + h[0] / float(k),) + tuple(h[1:]) for h, k, b in zip(hits, nh, big)]


def set_order_sums(feats, masses, hit_class, n_class, ref_ids=None, order="set"):
    """Python restatement of ExonBin::read_count: per class the first-inserted hit of every key (ref_id, ((off, len), ...)),
    keys in tuple order (the same lexicographic and prefix rule as Contig::operator<), float32 sum one member at a time.
    order="hit" / "reverse" sum the same members in insertion / reverse set order instead (what a wrong order would give)."""
    members = [dict() for _ in range(n_class)]
    for h, c in enumerate(hit_class):
        if c < 0:
            continue
        key = (int(ref_ids[h]) if ref_ids is not None else 0, tuple((int(o), int(ln)) for _, o, ln in feats[h]))
        members[c].setdefault(key, (h, np.float32(masses[h])))
    out = []
    for m in members:
        if order == "set":
            vals = [m[k][1] for k in sorted(m)]
        elif order == "reverse":
            vals = [m[k][1] for k in sorted(m, reverse=True)]
        else:
            vals = [v for _, v in sorted(m.values(), key=lambda x: x[0])]
        s = np.float32(0.0)
        for v in vals:
            s = np.float32(s + v)
        out.append((s, len(m)))
    return out


def sweep(group=None):
    from strawberry_b200 import builder
    for s in range(160):
        if s % 17 == 0 or (group is not None and s % 3 != group):
            continue
        isoforms, hits, rl = locusgen.random_locus(s)
        hits = fractional(hits, s)
        tfe = [locusgen.transcript_features(ex) for ex in isoforms]
        hl = [(m, builder.pair_features(l, r)) for m, l, r in hits]
        yield s, isoforms, hits, rl, tfe, hl


def test_host_builder_sums_fractional_masses_in_set_order(oracle_mod, sbq_lib_path):
    from strawberry_b200 import builder
    n_cls = n_hit_order = n_reverse = 0
    for s, isoforms, hits, rl, tfe, hl in sweep():
        spec = specs_for(s, hits)
        model = builder.Model.normal(spec[1], spec[2]) if spec[0] == "normal" else builder.Model.empirical(spec[1])
        host = builder.build_locus(tfe, hl, read_len=rl, model=model)
        feats, masses = [f for _, f in hl], [m for m, _ in hl]
        want = set_order_sums(feats, masses, host["hit_class"], len(host["classes"]))
        for c, (cl, (ms, nf)) in enumerate(zip(host["classes"], want)):
            assert np.float32(cl["mass"]) == ms and cl["count"] == int(ms) and cl["nfrag"] == nf, (s, c, cl, ms, nf)
        for order in ("hit", "reverse"):
            other = set_order_sums(feats, masses, host["hit_class"], len(host["classes"]), order=order)
            d = sum(a[0] != b[0] for a, b in zip(want, other))
            n_hit_order += d if order == "hit" else 0
            n_reverse += d if order == "reverse" else 0
        n_cls += len(want)
        if oracle_mod.have_ref() and s % 5 == 0:
            ref = reference_table(oracle_mod, isoforms, hits, rl, spec)
            assert len(ref["classes"]) == len(want)
            for c, (rc, (ms, nf)) in enumerate(zip(ref["classes"], want)):
                assert np.float32(rc["count_f"]) == ms and rc["count"] == int(ms) and rc["nfrags"] == nf, (s, c)
    # the inputs must tell the orders apart, or the test could not catch a wrong one
    assert n_cls > 1000 and n_hit_order > 20 and n_reverse > 300, (n_cls, n_hit_order, n_reverse)


# ---------------------------------------------------------------------------------------------------------------- GPU
def device_tables(loci, model, read_len, mode, ref_ids=None):
    """One raw batch in the given mass mode -> per-locus dicts in the shape builder.build_locus returns (as in
    test_gpu_rawbuild.device_tables). ref_ids: None, or per locus the hits' ref ids."""
    from strawberry_b200 import api, builder
    q = api.Quantifier()
    q.set_insert_model(model, read_len)
    builder.set_raw_mass_mode(q, mode)
    for l, (tfe, hl) in enumerate(loci):
        builder.submit_raw(q, tfe, hl, read_len=read_len, ref_ids=ref_ids[l] if ref_ids else None)
    q.upload()
    n_hit = sum(len(hl) for _, hl in loci)
    cls, coords, b = builder.fetch_raw_classes(q, n_hit), builder.fetch_raw_coords(q, n_hit), q.fetch_batch()
    out, h0 = [], 0
    for l, (tfe, hl) in enumerate(loci):
        r0, r1 = int(b["loc_row_off"][l]), int(b["loc_row_off"][l + 1])
        k0, k1 = int(b["row_ptr"][r0]), int(b["row_ptr"][r1])
        classes = [dict(coords=[int(x) for x in coords[int(cls["class_rep"][c])]], count=int(b["count"][c]), mass=float(cls["class_mass"][c]),
                        nfrag=int(cls["class_nfrag"][c])) for c in range(r0, r1)]
        out.append(dict(classes=classes, row_ptr=b["row_ptr"][r0:r1 + 1] - k0, col=b["col"][k0:k1], alpha=b["alpha"][k0:k1],
                        hit_class=cls["hit_class"][h0:h0 + len(hl)], iso_len=b["iso_len"][int(b["loc_iso_off"][l]):int(b["loc_iso_off"][l + 1])]))
        h0 += len(hl)
    return q, out


def host_table(tfe, hl, rl, model, ref_ids=None):
    from strawberry_b200 import builder
    return builder.build_locus(tfe, hl, read_len=rl, model=model, ref_ids=ref_ids)


@pytest.mark.gpu
@pytest.mark.parametrize("group", [0, 1, 2])
def test_device_any_mode_matches_host_builder_on_the_sweep(sbq_lib_path, group):
    from strawberry_b200 import builder
    from test_gpu_rawbuild import assert_same_table
    by_key = {}
    for s, isoforms, hits, rl, tfe, hl in sweep(group):
        spec = specs_for(s, hits)
        key = (rl,) + ((spec[0], spec[1], spec[2]) if spec[0] == "normal" else ("emp", s))
        by_key.setdefault(key, []).append((s, rl, tfe, hl, spec))
    n_frac = 0
    for items in by_key.values():
        spec, rl = items[0][4], items[0][1]
        model = builder.Model.normal(spec[1], spec[2]) if spec[0] == "normal" else builder.Model.empirical(spec[1])
        q, dev = device_tables([(it[2], it[3]) for it in items], model, rl, builder.RAW_MASS_ANY)
        q.close()
        for it, d in zip(items, dev):
            host = host_table(it[2], it[3], rl, model)
            assert_same_table(d, host, f"seed {it[0]}")
            n_frac += sum(c["mass"] != int(c["mass"]) for c in host["classes"])
    assert n_frac > 100


def adversarial_locus(seed):
    """Classes whose members tie on their first one to three features and differ deeper, single-end lists that are prefixes of
    paired ones, code-blind duplicates (5S50M variants) with another fractional mass, exact duplicates, mixed ref ids, and a
    few large members among 1/3, 1/7, ... fractions. Hits sorted by their first offset, like HitCluster::uniq_hits()."""
    from strawberry_b200 import builder
    rng = np.random.default_rng(seed)
    tfe = [locusgen.transcript_features([(1001, 6000)]), locusgen.transcript_features([(1001, 2000), (3001, 6000)])]
    fracs = [1 / 3, 1 / 7, 1 / 5, 1 / 6, 0.1, 2 / 3, 3 / 7]
    hl, refs = [], []

    def mass():
        return BIG if rng.random() < 0.03 else float(rng.choice(fracs)) * int(rng.integers(1, 4))
    for _ in range(1500):
        kind = rng.random()
        if kind < 0.7:                                           # MATCH / GAP lists from few offsets and lengths: deep ties
            off, feats = int(rng.choice([1100, 1101, 1180, 3100])), []
            nb = int(rng.integers(1, 5))
            for k in range(nb):
                ln = int(rng.choice([20, 21]))
                feats.append((0, off, ln))
                off += ln
                if k + 1 < nb:
                    g = int(rng.choice([10, 11, 30]))
                    feats.append((2, off, g))
                    off += g
            hl.append((mass(), feats))
        else:                                                    # mate pairs, the left mate sometimes soft-clipped (same _frags element)
            p = int(rng.choice([1050, 1060, 3200]))
            left = (p, [(4, 5), (0, 50)] if rng.random() < 0.5 else [(0, 50)])
            right = (p + int(rng.choice([70, 90])), [(0, 50)]) if rng.random() < 0.8 else None
            hl.append((mass(), builder.pair_features(left, right)))
        refs.append(int(rng.choice([0, 0, 1, 3])))
    order = sorted(range(len(hl)), key=lambda h: (hl[h][1][0][1] if hl[h][1] else 0))
    return tfe, [hl[h] for h in order], [refs[h] for h in order]


@pytest.mark.gpu
def test_device_any_mode_adversarial_classes_and_shuffled_submit(sbq_lib_path):
    from strawberry_b200 import builder
    from test_gpu_rawbuild import assert_same_table
    model = builder.Model.normal(200.0, 40.0)
    loci, refs = [], []
    for seed in (7, 8):
        tfe, hl, rid = adversarial_locus(seed)
        perm = np.random.default_rng(seed).permutation(len(hl))
        loci += [(tfe, hl), (tfe, [hl[i] for i in perm])]          # the same locus, its hits submitted in another order
        refs += [rid, [rid[i] for i in perm]]
    q, dev = device_tables(loci, model, 50, builder.RAW_MASS_ANY, ref_ids=refs)
    q.close()
    n_dup = n_order = 0
    for (tfe, hl), rid, d in zip(loci, refs, dev):
        host = host_table(tfe, hl, 50, model, ref_ids=rid)
        assert_same_table(d, host, "adversarial locus")
        feats, masses = [f for _, f in hl], [m for m, _ in hl]
        n_dup += int((host["hit_class"] >= 0).sum()) - sum(c["nfrag"] for c in host["classes"])   # members whose mass does not count
        want = set_order_sums(feats, masses, host["hit_class"], len(host["classes"]), ref_ids=rid)
        other = set_order_sums(feats, masses, host["hit_class"], len(host["classes"]), ref_ids=rid, order="hit")
        assert [np.float32(c["mass"]) for c in d["classes"]] == [w[0] for w in want]
        n_order += sum(a[0] != b[0] for a, b in zip(want, other))
    assert n_dup > 100 and n_order > 0, (n_dup, n_order)


@pytest.mark.gpu
def test_device_any_mode_big_loci_and_em(oracle_mod, sbq_lib_path):
    """The three >= 10 000-hit loci of test_gpu_rawbuild.test_device_class_tables_big_loci_and_em with 1/NH masses: device
    table == host table; the EM on the device-built batch == the oracle on the host-built CSR."""
    from strawberry_b200 import builder, synth
    from test_gpu_rawbuild import assert_same_table, inputs
    from util import assert_matches_oracle
    model = builder.Model.normal(220.0, 40.0)
    rl, loci = 50, []
    for seed in (1001, 1002, 1003):
        isoforms, _, _, tfe, _ = inputs(seed, max_exon=14, max_iso=9, max_frag=50)
        hits = fractional(locusgen.make_hits(np.random.default_rng(seed), isoforms, 60000, rl, frag_mean=220, frag_sd=40, noise=True), seed)
        loci.append((tfe, [(m, builder.pair_features(l, r)) for m, l, r in hits]))
    assert max(len(h) for _, h in loci) >= 10000
    q, dev = device_tables(loci, model, rl, builder.RAW_MASS_ANY)
    parts = []
    for (tfe, hl), d in zip(loci, dev):
        host = host_table(tfe, hl, rl, model)
        assert_same_table(d, host, f"big locus with {len(hl)} hits")
        parts.append(dict(loc_row_off=np.array([0, len(host["count"])]), loc_iso_off=np.array([0, host["n_iso"]]), row_ptr=host["row_ptr"], col=host["col"],
                          alpha=host["alpha"], count=host["count"], iso_len=host["iso_len"], total_mapped_reads=1_000_000))
    b = synth.concat(parts)
    q.solve(1_000_000)
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    res = q.results()
    q.close()
    assert_matches_oracle(res, oracle_mod.quantify_batch(b, 1_000_000), b, "EM on the device-built class table (1/NH masses)")


@pytest.mark.gpu
def test_any_mode_equals_default_mode_on_integer_masses(sbq_lib_path):
    from strawberry_b200 import api, builder
    loci = []
    for seed in range(200, 260):
        isoforms, hits, _ = locusgen.random_locus(seed)
        loci.append(([locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits]))
    n_hit = sum(len(hl) for _, hl in loci)
    out = []
    for mode in (builder.RAW_MASS_HALVES, builder.RAW_MASS_ANY):
        q = api.Quantifier()
        q.set_insert_model(builder.Model.normal(220.0, 40.0), 50)
        builder.set_raw_mass_mode(q, mode)
        for tfe, hl in loci:
            builder.submit_raw(q, tfe, hl, read_len=50)
        q.upload()
        out.append((q.fetch_batch(), builder.fetch_raw_classes(q, n_hit), builder.fetch_raw_coords(q, n_hit)))
        q.close()
    (b0, c0, x0), (b1, c1, x1) = out
    for k in b0:
        assert np.array_equal(b0[k], b1[k]), k
    for k in c0:
        assert np.array_equal(c0[k], c1[k]), k
    assert all(np.array_equal(u, v) for u, v in zip(x0, x1))


@pytest.mark.gpu
def test_any_mode_on_two_gpus_matches_one():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from strawberry_b200 import api, builder
    loci = []
    for seed in range(40, 64):
        isoforms, hits, _ = locusgen.random_locus(seed)
        hits = fractional(hits, seed)
        loci.append(([locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits]))
    out = []
    for n in (1, 2):
        q = api.Quantifier(device=0, n_gpus=n, min_iso_frac=0.01)
        q.set_insert_model(builder.Model.normal(200.0, 40.0), 50)
        builder.set_raw_mass_mode(q, builder.RAW_MASS_ANY)
        for tfe, hl in loci:
            builder.submit_raw(q, tfe, hl, read_len=50)
        q.run(250_000)
        out.append((q.results(), q.locus_devices(), q.stats()))
        q.close()
    (ref, _, st1), (got, dev, st2) = out
    for k in ("theta", "fpkm", "frac", "keep", "iters", "status"):
        assert np.array_equal(got[k], ref[k], equal_nan=True), k
    assert np.allclose(got["tpm"], ref["tpm"], rtol=1e-12, equal_nan=True)
    assert sorted(set(dev.tolist())) == [0, 1]
    assert st2["n_loci"] == st1["n_loci"] == len(loci) and st2["nnz"] == st1["nnz"] and st2["n_row"] == st1["n_row"]


@pytest.mark.gpu
def test_mass_mode_setter_and_any_mode_refusals(sbq_lib_path):
    from strawberry_b200 import api, builder
    isoforms, hits, rl = locusgen.random_locus(5)
    tfe = [locusgen.transcript_features(ex) for ex in isoforms]
    hl = [(m / 3.0, builder.pair_features(l, r)) for m, l, r in hits]
    q = api.Quantifier()
    for bad in (2, -1):
        with pytest.raises(api.SbqError) as e:
            builder.set_raw_mass_mode(q, bad)
        assert e.value.code == api.SBQ_ERR_INVALID
    q.set_insert_model(builder.Model.normal(200.0, 40.0), rl)
    builder.set_raw_mass_mode(q, builder.RAW_MASS_ANY)
    builder.submit_raw(q, tfe, hl, read_len=rl)
    q.upload()                                                   # fractional masses: accepted in ANY mode
    for h in range(len(hl)):                                     # the first hit that has a class
        if builder.fetch_raw_classes(q, len(hl))["hit_class"][h] >= 0:
            break
    for poison in (float("nan"), float("inf"), -0.5):
        q.clear()
        bad = list(hl)
        bad[h] = (poison, bad[h][1])
        builder.submit_raw(q, tfe, bad, read_len=rl)
        with pytest.raises(api.SbqError) as e:
            q.upload()
        assert e.value.code == api.SBQ_ERR_UNSUPPORTED and "SBQ_RAW_MASS_ANY" in str(e.value), poison
    q.close()


# -------------------------------------------------------------------------------------------------------- integration
REFDIR = os.path.join(ROOT, "oracle", "_ref")


def write_multimapped_dataset(sam_path, gtf_path, n_genes=120, seed=1, read_len=75, frags_per_gene=(20, 400), multi_rate=0.25):
    """tests/samgen.py's layout (genes on one chromosome, paired-end M/N reads sampled from the isoforms, GTF transcript and exon
    lines) with multimapped fragments: about multi_rate of the fragments are also placed at one to three other genes; every
    alignment of such a fragment carries NH:i:k, the first one is primary and the others are flagged secondary (256)."""
    import samgen
    rng = np.random.default_rng(seed)
    genes, pos = [], 10_000
    for g in range(n_genes):
        isoforms = locusgen.make_gene(rng, int(rng.integers(2, 12)), int(min(12, np.ceil(rng.pareto(1.2) + 1))), exon_len=(90, 400),
                                      intron_len=(200, 1500), start=pos)
        isoforms = [ex for ex in isoforms if sum(r - l + 1 for l, r in ex) >= 2 * read_len + 20]
        if not isoforms:
            continue
        genes.append(isoforms)
        pos = max(r for ex in isoforms for _, r in ex) + 5_000
    chrom_len = pos + 10_000

    def place(isoforms):
        """one fragment from a random isoform of the gene: (left mate, right mate) as (pos, ops), or None"""
        t = int(rng.integers(0, len(isoforms)))
        L = sum(r - l + 1 for l, r in isoforms[t])
        fl = int(np.clip(rng.normal(250, 30), read_len + 1, L))
        s = int(rng.integers(0, L - fl + 1))
        lb = locusgen._blocks(isoforms[t], s, s + read_len)
        rb = locusgen._blocks(isoforms[t], s + fl - read_len, s + fl)
        if lb[0][0] == rb[0][0]:
            return None                               # mates starting at the same position are discarded by the reference
        return locusgen._cigar(lb, rng, noise=False), locusgen._cigar(rb, rng, noise=False), rb[-1][1]

    recs, rid = [], 0
    with open(gtf_path, "w") as gtf:
        for g, isoforms in enumerate(genes):
            for t, exons in enumerate(isoforms):
                attr = f'gene_id "G{g}"; transcript_id "G{g}.T{t}";'
                gtf.write(f"chr1\tsynth\ttranscript\t{exons[0][0]}\t{exons[-1][1]}\t.\t+\t.\t{attr}\n")
                for (el, er) in exons:
                    gtf.write(f"chr1\tsynth\texon\t{el}\t{er}\t.\t+\t.\t{attr}\n")
    for g in range(len(genes)):
        for _ in range(int(rng.integers(*frags_per_gene))):
            where = [g]
            if rng.random() < multi_rate:
                others = [x for x in range(len(genes)) if x != g]
                where += [int(x) for x in rng.choice(others, int(rng.integers(1, 4)), replace=False)]
            alns = [a for a in (place(genes[x]) for x in where) if a is not None]
            if not alns:
                continue
            name = f"r{rid}"
            rid += 1
            for k, ((lpos, lops), (rpos, rops), rend) in enumerate(alns):
                sec = 256 if k else 0
                tlen = rend - lpos + 1
                for pos_, ops, flag, mpos, tl in ((lpos, lops, 99 | sec, rpos, tlen), (rpos, rops, 147 | sec, lpos, -tlen)):
                    tags = f"NH:i:{len(alns)}" + ("\tXS:A:+" if any(o == 3 for o, _ in ops) else "")
                    recs.append((pos_, f"{name}\t{flag}\tchr1\t{pos_}\t255\t{samgen._cigar_str(ops)}\t=\t{mpos}\t{tl}\t{'A' * read_len}\t{'I' * read_len}\t{tags}\n"))
    recs.sort(key=lambda x: x[0])
    with open(sam_path, "w") as sam:
        sam.write("@HD\tVN:1.0\tSO:coordinate\n")
        sam.write(f"@SQ\tSN:chr1\tLN:{chrom_len}\n")
        for _, line in recs:
            sam.write(line)
    return dict(n_genes=len(genes), n_isoforms=sum(len(g) for g in genes))


@pytest.mark.gpu
def test_batched_dropin_with_multimapped_hits_matches_reference(tmp_path):
    """strawberry_sbq_batched --allow-multimapped-hits against the unmodified reference binary: GTF records byte-identical with
    -p 1 (in order), theta log lines identical, and the class tables built on the device (SBQ_TIMING report)."""
    import subprocess
    from test_gpu_integration import gtf_body, theta_lines
    ref_bin, batched, samtools = (os.path.join(REFDIR, b) for b in ("strawberry_ref", "strawberry_sbq_batched", "samtools_ref"))
    if not all(os.path.exists(b) for b in (ref_bin, batched, samtools)):
        pytest.skip("oracle/_ref binaries not built (make -C integration)")
    sam, gtf, bam = (str(tmp_path / n) for n in ("s.sam", "s.gtf", "s.bam"))
    info = write_multimapped_dataset(sam, gtf, seed=11)
    with open(bam, "wb") as fh:
        subprocess.run([samtools, "view", "-bS", sam], check=True, stdout=fh, stderr=subprocess.DEVNULL)
    outs = {}
    for tag, binary in (("ref", ref_bin), ("sbq", batched)):
        out, log = str(tmp_path / f"{tag}.gtf"), str(tmp_path / f"{tag}.log")
        r = subprocess.run([binary, bam, "-g", gtf, "-r", "-o", out, "-T", log, "-p", "1", "--allow-multimapped-hits"], check=True,
                           stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, timeout=600, env=dict(os.environ, SBQ_TIMING="1"))
        outs[tag] = (gtf_body(out), theta_lines(log), [l for l in r.stderr.splitlines() if l.startswith("SBQ_TIMING")])
    (ref_gtf, ref_theta, _), (got_gtf, got_theta, timing) = outs["ref"], outs["sbq"]
    assert len(ref_gtf) > info["n_isoforms"] and len(ref_theta) > 50
    assert got_gtf == ref_gtf, "GTF records differ from the reference (byte diff, -p 1, in order)"
    assert got_theta == ref_theta, "theta log lines differ from the reference"
    fields = timing[-1].split()
    assert int(fields[fields.index("device_class_loci") + 1]) == int(fields[fields.index("loci") + 1]) > 0, timing
