"""Device class-table build (sbq_submit_raw + sbq_upload) on seeded raw batches: time per upload, and the device tables of
two libsbq.so builds compared on the short-read batch.

Batches:
  short  4000 loci of the tests/test_builder.py sweep (tests/locusgen.random_locus), read length 50, normal(220, 40) inserts:
         the human-shaped short-read case, where every hit touches at most 16 segments and every class spans at most 32
  long   200 full-length long-read loci (40-exon genes, one 1500 bp read per fragment), long-read mode: every class touches
         more than 16 segments
  multimapped  the short batch with every mass m replaced by m / NH (NH seeded from 2..8), as --allow-multimapped-hits gives,
         uploaded in SBQ_RAW_MASS_ANY mode: class masses summed in the reference's set order on the device

  python tools/rawbuild_bench.py --lib new=strawberry_b200/libsbq.so --lib parent=/path/to/parent/strawberry_b200/libsbq.so --out DIR
      every upload leg runs in a child process of its own (SBQ_LIB_PATH selects the library, and the strawberry_b200 package
      next to it is imported when there is one); the legs alternate between the
      libraries for --rounds rounds, each leg times --uploads uploads of the same batch after --warmup untimed ones
      (median and spread of the stats' upload_ms / weights_ms and of the host wall time of sbq_upload); the short-read tables
      of every library are checked equal to the first one's. A library that refuses a batch (the long-read one, or the
      multimapped one when it has no SBQ_RAW_MASS_ANY) is reported as such.
  python tools/rawbuild_bench.py --shapes
      no GPU: the device memory the descriptors of both batches take, old fixed layout ([H][16] coordinates, 32-slot pool per
      CSR entry) against the variable-length one, counted from the host builder's tables.
"""
import argparse
import bisect
import json
import os
import pickle
import subprocess
import sys
import tempfile

import numpy as np

KINDS = ("short", "long", "multimapped")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def make_batch(kind):
    import locusgen
    from strawberry_b200 import builder
    loci = []
    if kind in ("short", "multimapped"):
        rng = np.random.default_rng(30_000)
        for seed in range(4000):
            isoforms, hits, _ = locusgen.random_locus(10_000 + seed)
            if kind == "multimapped":
                hits = [(m / float(nh), l, r) for (m, l, r), nh in zip(hits, rng.integers(2, 9, len(hits)))]
            loci.append(([locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits]))
        return dict(loci=loci, read_len=50, mean=220.0, sd=40.0, long_read=False, mass_any=kind == "multimapped")
    for seed in range(200):
        rng = np.random.default_rng(20_000 + seed)
        isoforms = locusgen.make_gene(rng, 40, 6, exon_len=(40, 160), intron_len=(100, 600))
        hits = locusgen.make_hits(rng, isoforms, 300, 1500, frag_mean=1500, frag_sd=1, noise=False, single_rate=1.0)
        loci.append(([locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits]))
    return dict(loci=loci, read_len=1500, mean=1500.0, sd=1.0, long_read=True)


def child(batch_path, uploads, warmup, dump):
    """one leg: submit the batch once, upload it warmup + uploads times; print JSON, optionally dump the device tables"""
    import time
    tree = os.path.dirname(os.path.dirname(os.environ["SBQ_LIB_PATH"]))
    if os.path.exists(os.path.join(tree, "strawberry_b200", "__init__.py")):
        sys.path.insert(0, tree)   # the Python binding of the library's own checkout: an older one lacks newer symbols
    from strawberry_b200 import api, builder
    bt = pickle.load(open(batch_path, "rb"))
    q = api.Quantifier(device=0)
    q.set_insert_model(builder.Model.normal(bt["mean"], bt["sd"]), bt["read_len"])
    if bt.get("mass_any"):
        if not hasattr(builder, "set_raw_mass_mode"):
            print(json.dumps(dict(refused=api.SBQ_ERR_UNSUPPORTED, message="this library has no sbq_set_raw_mass_mode")))
            return
        builder.set_raw_mass_mode(q, builder.RAW_MASS_ANY)
    for tfe, hl in bt["loci"]:
        builder.submit_raw(q, tfe, hl, read_len=bt["read_len"], long_read=bt["long_read"])
    up, wt, wall = [], [], []
    try:
        for k in range(warmup + uploads):
            t0 = time.perf_counter()
            q.upload()
            t1 = time.perf_counter()
            if k >= warmup:
                st = q.stats()
                up.append(st["upload_ms"]), wt.append(st["weights_ms"]), wall.append((t1 - t0) * 1e3)
    except api.SbqError as e:
        print(json.dumps(dict(refused=e.code, message=str(e))))
        return
    st = q.stats()
    if dump:
        n_hit = sum(len(hl) for _, hl in bt["loci"])
        b, cls = q.fetch_batch(), builder.fetch_raw_classes(q, n_hit)
        coords = np.concatenate([c[:n] for c, n in zip(cls["coords"], cls["ncoord"])])   # slots past the count are not defined in older builds
        np.savez(dump, coords=coords, **{k: v for k, v in b.items()}, **{k: v for k, v in cls.items() if k != "coords"})
    q.close()
    print(json.dumps(dict(upload_ms=up, weights_ms=wt, wall_ms=wall, n_loci=st["n_loci"], n_row=st["n_row"], nnz=st["nnz"], n_hit=sum(len(h) for _, h in bt["loci"]))))


def summary(xs):
    xs = np.asarray(xs, float)
    return dict(median=float(np.median(xs)), min=float(xs.min()), max=float(xs.max()), n=len(xs))


def shapes():
    """device bytes of the coordinate lists and weight descriptors: fixed layout (before) against variable-length (now)"""
    from strawberry_b200 import builder
    out = {}
    for kind in ("short", "long"):
        bt = make_batch(kind)
        model = builder.Model.normal(bt["mean"], bt["sd"])
        H = n_coord = nnz = R = n_seg = 0
        for tfe, hl in bt["loci"]:
            tb = builder.build_locus(tfe, hl, read_len=bt["read_len"], model=model, long_read=bt["long_read"])
            H += len(hl)
            R += len(tb["classes"])
            nnz += len(tb["col"])
            for h, c in enumerate(tb["hit_class"]):
                n_coord += len(tb["classes"][c]["coords"]) if c >= 0 else 0
            if not bt["long_read"]:
                for c, cl in enumerate(tb["classes"]):
                    for k in range(tb["row_ptr"][c], tb["row_ptr"][c + 1]):
                        isg = tb["iso_segs"][int(tb["col"][k])]
                        n_seg += bisect.bisect_left(isg, cl["coords"][-1]) - bisect.bisect_left(isg, cl["coords"][0]) + 1
        out[kind] = dict(n_hit=H, n_class=R, nnz=nnz, n_coord_classified_hits=n_coord, n_spanned_segments=n_seg,
                         # [H][16] u16 + u8 count, against u32 count + i64 offset per hit + u16 per coordinate (classified hits only
                         # are counted here; a hit compatible with no isoform also keeps its list)
                         hit_bytes_fixed=H * 33, hit_bytes_variable=H * 12 + 8 + 2 * n_coord,
                         # 32 x u32 pool + u8 count per entry, against u32 per spanned segment + u16 count per entry + i32 count and
                         # i64 offset per class
                         desc_bytes_fixed=nnz * 129, desc_bytes_variable=4 * n_seg + 2 * nnz + 12 * R + 8)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--lib", action="append", default=[], help="NAME=PATH of a libsbq.so (repeat; the first is the reference for the table check)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--uploads", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for rawbuild_bench.json")
    ap.add_argument("--shapes", action="store_true")
    ap.add_argument("--child", nargs=4, metavar=("BATCH", "UPLOADS", "WARMUP", "DUMP"), help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        return child(a.child[0], int(a.child[1]), int(a.child[2]), a.child[3] if a.child[3] != "-" else None)
    if a.shapes:
        print(json.dumps(shapes(), indent=1))
        return
    if not a.lib:
        ap.error("--lib NAME=PATH is required")
    libs = [tuple(x.split("=", 1)) for x in a.lib]
    res = dict(gpu=subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                  capture_output=True, text=True).stdout.strip().splitlines()[:1], legs=[])
    with tempfile.TemporaryDirectory() as tmp:
        paths = {}
        for kind in KINDS:
            paths[kind] = os.path.join(tmp, f"{kind}.pkl")
            pickle.dump(make_batch(kind), open(paths[kind], "wb"))
        timings = {(n, k): dict(upload_ms=[], weights_ms=[], wall_ms=[], per_leg_median_upload_ms=[]) for n, _ in libs for k in paths}
        refused = {}
        for r in range(a.rounds):
            for kind in KINDS:
                for name, path in libs:
                    dump = os.path.join(tmp, f"{name}.npz") if kind == "short" and r == 0 else "-"
                    env = dict(os.environ, SBQ_LIB_PATH=os.path.abspath(path))
                    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", paths[kind], str(a.uploads), str(a.warmup), dump],
                                       capture_output=True, text=True, env=env)
                    if p.returncode:
                        raise RuntimeError(f"{name} {kind}: {p.stderr[-2000:]}")
                    leg = json.loads(p.stdout.strip().splitlines()[-1])
                    res["legs"].append(dict(round=r, kind=kind, lib=name, **leg))
                    if "refused" in leg:
                        refused[(name, kind)] = leg["message"]
                        continue
                    t = timings[(name, kind)]
                    for k in ("upload_ms", "weights_ms", "wall_ms"):
                        t[k] += leg[k]
                    t["per_leg_median_upload_ms"].append(float(np.median(leg["upload_ms"])))
                    t["shape"] = dict(n_loci=leg["n_loci"], n_hit=leg["n_hit"], n_row=leg["n_row"], nnz=leg["nnz"])
        ref_name = libs[0][0]
        ref = np.load(os.path.join(tmp, f"{ref_name}.npz"))
        same = {}
        for name, _ in libs[1:]:
            got = np.load(os.path.join(tmp, f"{name}.npz"))
            same[name] = {k: bool(ref[k].shape == got[k].shape and np.array_equal(ref[k], got[k])) for k in ref.files}
    res["summary"] = {f"{n}/{k}": (dict(refused=refused[(n, k)]) if (n, k) in refused else
                                   dict(shape=v.get("shape"), **{m: summary(v[m]) for m in ("upload_ms", "weights_ms", "wall_ms")},
                                        per_leg_median_upload_ms=v["per_leg_median_upload_ms"]))
                      for (n, k), v in timings.items()}
    res["short_tables_equal_to_" + ref_name] = same
    text = json.dumps(res, indent=1)
    print(json.dumps(dict(gpu=res["gpu"], summary=res["summary"], tables=same), indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "rawbuild_bench.json"), "w").write(text)
    bad = [n for n, d in same.items() if not all(d.values())]
    if bad:
        sys.exit(f"device tables differ from {ref_name}'s on the short-read batch: {bad} {same}")


if __name__ == "__main__":
    main()
