"""GPU: device class assignment (sbq_submit_raw) on the two shapes that need variable-length lists - long reads, whose hits
touch every segment of a gene (here 17 to 70+ segments per hit), and exon-dense loci with long inserts, whose classes span
more than 32 (and more than 54) segments of an isoform - against the host builder: classes with their FULL coordinate lists
(sbq_fetch_raw_coords), the class of every hit, counts, float masses, the CSR and alpha (<= 1e-12 relative); the EM on a
device-built long-read locus of 10 000+ hits against the oracle; two GPUs against one; and, where it is built, the compiled
reference."""
import bisect
import os
import subprocess

import numpy as np
import pytest

import locusgen
from test_gpu_rawbuild import assert_same_table, device_tables, inputs

pytestmark = pytest.mark.gpu


def long_read_locus(seed, n_frag=300, n_exon=40, n_iso=6, exon_len=(40, 160)):
    """A full-length long-read locus: one 1500 bp single read per fragment."""
    from strawberry_b200 import builder
    rng = np.random.default_rng(seed)
    isoforms = locusgen.make_gene(rng, n_exon, n_iso, exon_len=exon_len, intron_len=(100, 600))
    hits = locusgen.make_hits(rng, isoforms, n_frag, 1500, frag_mean=1500, frag_sd=1, noise=False, single_rate=1.0)
    return isoforms, hits, [locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits]


def dense_locus(seed):
    """Tiny exons (6-16 bp) and inserts of 900 +- 300 bp: 50 bp mates whose classes span up to ~70 segments of an isoform."""
    from strawberry_b200 import builder
    rng = np.random.default_rng(seed)
    isoforms = locusgen.make_gene(rng, 90, 5, exon_len=(6, 16), intron_len=(30, 80))
    hits = locusgen.make_hits(rng, isoforms, 400, 50, frag_mean=900, frag_sd=300, noise=False)
    return isoforms, hits, [locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits]


def with_full_coords(q, dev, loci):
    """device_tables keeps the first 16 coordinates of a class: put the representative's full list (sbq_fetch_raw_coords)
    in their place, and check that every classified hit's own list is its class's list and that sbq_fetch_raw_classes
    reports the first 16 of each list with the count saturated at 255."""
    from strawberry_b200 import builder
    n_hit = sum(len(hl) for _, hl in loci)
    coords = builder.fetch_raw_coords(q, n_hit)
    cls = builder.fetch_raw_classes(q, n_hit)
    for h, full in enumerate(coords):
        n = len(full)
        assert cls["ncoord"][h] == min(n, 255)
        assert np.array_equal(cls["coords"][h][:min(n, 16)], full[:16]) and not cls["coords"][h][min(n, 16):].any()
    r, h0 = 0, 0
    for d, (_, hl) in zip(dev, loci):
        for cl in d["classes"]:
            cl["coords"] = [int(x) for x in coords[int(cls["class_rep"][r])]]
            r += 1
        for h, c in enumerate(d["hit_class"]):
            if c >= 0:
                assert [int(x) for x in coords[h0 + h]] == d["classes"][c]["coords"]
        h0 += len(hl)
    return dev


def spans(host):
    """number of isoform segments each CSR entry of a host table spans (ExonBin::bin_under_iso)"""
    out = []
    for c, cl in enumerate(host["classes"]):
        for k in range(host["row_ptr"][c], host["row_ptr"][c + 1]):
            isg = host["iso_segs"][int(host["col"][k])]
            out.append(bisect.bisect_left(isg, cl["coords"][-1]) - bisect.bisect_left(isg, cl["coords"][0]) + 1)
    return np.asarray(out)


def test_long_reads_with_sweep_loci_in_one_batch(sbq_lib_path):
    """30 long-read loci (every class touches more than 16 segments) and 30 loci of the ordinary sweep, one long-read batch."""
    from strawberry_b200 import builder
    model = builder.Model.normal(1500.0, 1.0)
    loci = [long_read_locus(s)[2:] for s in range(30)] + [inputs(s)[3:] for s in range(1, 160, 5)][:30]
    q, dev = device_tables(loci, model, 1500, long_read=True)
    dev = with_full_coords(q, dev, loci)
    q.close()
    widest = []
    for n, ((tfe, hl), d) in enumerate(zip(loci, dev)):
        host = builder.build_locus(tfe, hl, read_len=1500, model=model, long_read=True)
        assert_same_table(d, host, f"locus {n}")
        widest.append(max((len(c["coords"]) for c in host["classes"]), default=0))
    assert min(widest[:30]) > 16 and max(widest[:30]) > 30, widest[:30]


def test_exon_dense_classes_spanning_more_than_32_and_54_segments(sbq_lib_path):
    """alpha depends on effective_len here (pdf > 0 across the spans), on both sides of n = 54, where the reference's target
    mask (uint32_t)(uint64_t)(pow(2, n) - 1) turns from all ones to 0."""
    from strawberry_b200 import builder
    model = builder.Model.normal(900.0, 300.0)
    loci = [dense_locus(s)[2:] for s in (100, 101, 102, 103)]
    q, dev = device_tables(loci, model, 50)
    dev = with_full_coords(q, dev, loci)
    q.close()
    n_all, a_all = [], []
    for n, ((tfe, hl), d) in enumerate(zip(loci, dev)):
        host = builder.build_locus(tfe, hl, read_len=50, model=model)
        assert_same_table(d, host, f"dense locus {n}")
        n_all.append(spans(host))
        a_all.append(host["alpha"])
    ns, alpha = np.concatenate(n_all), np.concatenate(a_all)
    assert ((ns > 32) & (ns < 54) & (alpha > 0)).sum() >= 10       # weights of wide spans that the device must get right
    assert (ns >= 54).sum() >= 50 and (ns >= 64).sum() > 0
    assert ((ns <= 32) & (alpha > 0)).sum() > 100


def test_long_read_locus_of_10000_hits_and_em(oracle_mod, sbq_lib_path):
    from strawberry_b200 import api, builder, synth
    from util import assert_matches_oracle
    model = builder.Model.normal(1500.0, 1.0)
    _, _, tfe, hl = long_read_locus(7, n_frag=40000, n_exon=100, n_iso=12, exon_len=(30, 80))
    assert len(hl) >= 10000
    q, dev = device_tables([(tfe, hl)], model, 1500, long_read=True)
    dev = with_full_coords(q, dev, [(tfe, hl)])
    coords = builder.fetch_raw_coords(q, len(hl))
    assert min(len(c) for c in coords) > 16
    host = builder.build_locus(tfe, hl, read_len=1500, model=model, long_read=True)
    assert_same_table(dev[0], host, f"long-read locus with {len(hl)} hits")
    b = synth.concat([dict(loc_row_off=np.array([0, len(host["count"])]), loc_iso_off=np.array([0, host["n_iso"]]), row_ptr=host["row_ptr"],
                           col=host["col"], alpha=host["alpha"], count=host["count"], iso_len=host["iso_len"], total_mapped_reads=1_000_000)])
    q.solve(1_000_000)
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    res = q.results()
    q.close()
    assert_matches_oracle(res, oracle_mod.quantify_batch(b, 1_000_000), b, "EM on the device-built long-read table")


@pytest.mark.parametrize("kind", ["long", "dense"])
def test_two_gpus_match_one(kind):
    """n_gpus = 2 in one context against one GPU: bitwise equal (theta / FPKM / frac / keep / iters / status)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from strawberry_b200 import api, builder
    if kind == "long":
        loci, rl, model = [long_read_locus(s)[2:] for s in range(12)], 1500, builder.Model.normal(1500.0, 1.0)
    else:
        loci, rl, model = [dense_locus(s)[2:] for s in range(100, 108)], 50, builder.Model.normal(900.0, 300.0)
    out = []
    for n in (1, 2):
        q = api.Quantifier(device=0, n_gpus=n, min_iso_frac=0.01)
        q.set_insert_model(model, rl)
        for tfe, hl in loci:
            builder.submit_raw(q, tfe, hl, read_len=rl, long_read=kind == "long")
        q.run(250_000)
        out.append((q.results(), q.locus_devices()))
        q.close()
    (ref, _), (got, dev) = out
    for k in ("theta", "fpkm", "frac", "keep", "iters", "status"):
        assert np.array_equal(got[k], ref[k], equal_nan=True), k
    assert sorted(set(dev.tolist())) == [0, 1]


def test_against_the_compiled_reference(oracle_mod, sbq_lib_path):
    if not oracle_mod.have_ref():
        pytest.skip("oracle/_ref/libsbref.so not built")
    from strawberry_b200 import builder
    for kind, seed in (("long", 0), ("long", 1), ("dense", 100), ("dense", 101)):
        isoforms, hits, tfe, hl = long_read_locus(seed) if kind == "long" else dense_locus(seed)
        rl, mean, sd = (1500, 1500.0, 1.0) if kind == "long" else (50, 900.0, 300.0)
        q, dev = device_tables([(tfe, hl)], builder.Model.normal(mean, sd), rl, long_read=kind == "long")
        dev = with_full_coords(q, dev, [(tfe, hl)])[0]
        q.close()
        ref = oracle_mod.ref_locus_context(tfe, hits, read_len=rl, long_read=kind == "long", total_mapped_reads=100000, mean=mean, sd=sd)
        segs = builder.build_locus(tfe, hl, read_len=rl, model=builder.Model.normal(mean, sd), long_read=kind == "long")["segs"]
        assert len(ref["classes"]) == len(dev["classes"]), (kind, seed)
        for c, rc in enumerate(ref["classes"]):
            d = dev["classes"][c]
            assert [list(segs[s]) for s in d["coords"]] == rc["coords"], (kind, seed, c)
            assert d["nfrag"] == rc["nfrags"] and d["count"] == rc["count"] and np.float32(d["mass"]) == np.float32(rc["count_f"]), (kind, seed, c)
            for k in range(dev["row_ptr"][c], dev["row_ptr"][c + 1]):
                w, w_ref = float(dev["alpha"][k]), rc["weights"][str(int(dev["col"][k]))]
                assert abs(w - w_ref) <= 1e-12 * max(abs(w_ref), 1e-300), (kind, seed, c, k)


def write_long_read_dataset(sam_path, gtf_path, n_genes=40, seed=5):
    """Single-end full-length reads of 1050-1800 bp (more than 10 distinct lengths above 1000 bp, so the reference switches to
    long-read mode) from genes of 24 exons, coordinate-sorted SAM + GTF."""
    import samgen
    rng = np.random.default_rng(seed)
    genes, pos = [], 10_000
    for _ in range(n_genes):
        isoforms = locusgen.make_gene(rng, 24, 4, exon_len=(60, 200), intron_len=(200, 1200), start=pos)
        isoforms = [ex for ex in isoforms if len(ex) >= 20 and sum(r - l + 1 for l, r in ex) >= 1900]
        if isoforms:
            genes.append(isoforms)
            pos = max(r for ex in isoforms for _, r in ex) + 5_000
    recs, rid = [], 0
    with open(gtf_path, "w") as gtf:
        for g, isoforms in enumerate(genes):
            for t, exons in enumerate(isoforms):
                attr = f'gene_id "G{g}"; transcript_id "G{g}.T{t}";'
                gtf.write(f"chr1\tsynth\ttranscript\t{exons[0][0]}\t{exons[-1][1]}\t.\t+\t.\t{attr}\n")
                for (el, er) in exons:
                    gtf.write(f"chr1\tsynth\texon\t{el}\t{er}\t.\t+\t.\t{attr}\n")
            lens = [sum(r - l + 1 for l, r in ex) for ex in isoforms]
            for _ in range(int(rng.integers(30, 200))):
                t = int(rng.integers(0, len(isoforms)))
                rl = int(rng.integers(1050, 1801))
                s = int(rng.integers(0, lens[t] - rl + 1))
                p, ops = locusgen._cigar(locusgen._blocks(isoforms[t], s, s + rl), rng, noise=False)
                tags = "NH:i:1" + ("\tXS:A:+" if any(o == 3 for o, _ in ops) else "")
                recs.append((p, f"r{rid}\t0\tchr1\t{p}\t255\t{samgen._cigar_str(ops)}\t*\t0\t0\t{'A' * rl}\t{'I' * rl}\t{tags}\n"))
                rid += 1
    recs.sort(key=lambda x: x[0])
    with open(sam_path, "w") as sam:
        sam.write(f"@HD\tVN:1.0\tSO:coordinate\n@SQ\tSN:chr1\tLN:{pos + 10_000}\n")
        for _, line in recs:
            sam.write(line)
    return len(genes)


def test_batched_dropin_on_long_reads_is_byte_exact(tmp_path):
    """The batched drop-in assigns classes on the GPU by default, long-read samples included: its GTF equals the reference's."""
    from test_gpu_integration import BATCHED, BINS, gtf_body, run
    if not all(os.path.exists(b) for b in BINS + [BATCHED]):
        pytest.skip("oracle/_ref binaries not built (make -C integration)")
    sam, gtf, bam = (str(tmp_path / n) for n in ("s.sam", "s.gtf", "s.bam"))
    assert write_long_read_dataset(sam, gtf) >= 20
    with open(bam, "wb") as fh:
        subprocess.run([BINS[2], "view", "-bS", sam], check=True, stdout=fh, stderr=subprocess.DEVNULL)
    outs = []
    for tag, binary in (("ref", BINS[0]), ("batched", BATCHED)):
        out = str(tmp_path / f"{tag}.gtf")
        run(binary, bam, gtf, out, str(tmp_path / f"{tag}.log"), 1)
        outs.append(gtf_body(out))
    assert len(outs[0]) > 20 and outs[1] == outs[0]
