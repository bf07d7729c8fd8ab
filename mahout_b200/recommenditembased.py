"""`mahout recommenditembased` on the GPU: upstream RecommenderJob (cf/taste/hadoop/item/) with the similarity phase
and the aggregate-and-recommend phase as native calls.

    python -m mahout_b200.recommenditembased --input prefs.csv --output recs.txt \
        --similarityClassname SIMILARITY_COSINE | SIMILARITY_SKETCH_COSINE [--numRecommendations 10] \
        [--maxPrefsPerUser 10] [--minPrefsPerUser 1] [--maxSimilaritiesPerItem 100] [--booleanData true] \
        [--threshold 0.1] [--usersFile ids.txt] [--itemsFile ids.txt] [--outputPathForSimilarityMatrix dir/part] \
        [--sketchWidth 4096] [--sketchDepth 4] [--sketchSeed 42] [--precision rescored|certified|tensor] \
        [--numGpus N]

Input `userID,itemID[,pref]` (tab or comma).  Output: `userID<TAB>[itemID:value,itemID:value,...]` per user with at
least one recommendation, users in ascending userID order, values as Float.toString writes them.  --usersFile and
--itemsFile hold one ID per line.  --maxPrefsInItemSimilarity and --randomSeed are accepted and do nothing (no
down-sampling takes place, as in itemsimilarity).  --filterFile, --userItemFile and --sequencefileOutput are not
supported.  Returns 0 on success, -1 on bad arguments or failure, like AbstractJob.

`--numGpus N` (0 = every visible GPU) runs the job on N GPUs of this process: the preparation on the first of them,
the similarity phase as one mb200_job_item_similarity call over all N (as itemsimilarity --numGpus), and the
recommend phase with the lists and user vectors replicated on every GPU and the users split between them
(multi.MultiItemBased).  The recommend phase returns the single-GPU bytes for any N; the similarity phase does so at
--precision rescored, so there the output file is the single-GPU job's byte for byte.
"""
from __future__ import annotations

import argparse
import sys
import time

import numpy as np

from . import itembased as ib
from . import similarity as sim
from .itemsimilarity import EXACT_MEASURES, MEASURES, _bool, multi_item_similarity, open_gpus

UNSUPPORTED = ("filterFile", "userItemFile", "sequencefileOutput")


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog="recommenditembased", add_help=True)
    ap.add_argument("--input", "-i", required=True)
    ap.add_argument("--output", "-o", required=True)
    ap.add_argument("--similarityClassname", "-s", required=True)
    ap.add_argument("--numRecommendations", type=int, default=ib.DEFAULT_NUM_RECOMMENDATIONS)
    ap.add_argument("--maxPrefsPerUser", type=int, default=ib.DEFAULT_MAX_PREFS_PER_USER)
    ap.add_argument("--minPrefsPerUser", "-mp", type=int, default=sim.DEFAULT_MIN_PREFS_PER_USER)
    ap.add_argument("--maxSimilaritiesPerItem", "-m", type=int, default=sim.DEFAULT_MAX_SIMILAR_ITEMS_PER_ITEM)
    ap.add_argument("--maxPrefsInItemSimilarity", type=int, default=500)
    ap.add_argument("--booleanData", "-b", default="false")
    ap.add_argument("--threshold", "-tr", type=float, default=None)
    ap.add_argument("--usersFile", default=None)
    ap.add_argument("--itemsFile", default=None)
    ap.add_argument("--outputPathForSimilarityMatrix", default=None)
    ap.add_argument("--randomSeed", type=int, default=None)
    ap.add_argument("--tempDir", default=None)
    ap.add_argument("--startPhase", type=int, default=0)
    ap.add_argument("--endPhase", type=int, default=2 ** 31 - 1)
    ap.add_argument("--sketchWidth", type=int, default=4096)
    ap.add_argument("--sketchDepth", type=int, default=4)
    ap.add_argument("--sketchSeed", type=int, default=42)
    ap.add_argument("--fracBits", type=int, default=1)
    ap.add_argument("--precision", default="rescored", choices=["rescored", "certified", "tensor"])
    ap.add_argument("--numGpus", type=int, default=None,
                    help="run the job on N GPUs of this process (0 = every visible GPU)")
    for name in UNSUPPORTED:
        ap.add_argument(f"--{name}", default=None)
    return ap


def format_line(user_id: int, items, values) -> str:
    """one line of the job's text output (RecommendedItemsWritable.toString)"""
    body = ",".join(f"{int(i)}:{sim.java_float_to_string(float(v))}" for i, v in zip(items, values))
    return f"{int(user_id)}\t[{body}]\n"


def _read_ids(path: str) -> list[int]:
    with open(path) as f:
        return [int(line.strip()) for line in f if line.strip()]


class RecommenderJob:
    def __init__(self):
        self.phase_s = {}   # wall clock of the phases of the last run, each ended by a device synchronise

    def run(self, argv) -> int:
        try:
            args = build_parser().parse_args(argv)
        except SystemExit:
            return -1
        for name in UNSUPPORTED:
            if getattr(args, name) is not None:
                print(f"recommenditembased: --{name} is not supported by the native job", file=sys.stderr)
                return -1
        if args.similarityClassname not in MEASURES:
            print(f"recommenditembased: the native path implements the cosine measure only "
                  f"(got {args.similarityClassname})", file=sys.stderr)
            return -1
        if not 1 <= args.numRecommendations <= ib.MAX_HOW_MANY:
            print(f"recommenditembased: --numRecommendations must be in [1, {ib.MAX_HOW_MANY}]", file=sys.stderr)
            return -1
        if args.maxPrefsPerUser < 1 or args.maxSimilaritiesPerItem < 1:
            print("recommenditembased: --maxPrefsPerUser and --maxSimilaritiesPerItem must be positive",
                  file=sys.stderr)
            return -1
        multi = None
        self.phase_s = {}
        try:
            import torch
            from . import ingest
            t0 = time.perf_counter()

            def phase(name):
                nonlocal t0
                torch.cuda.synchronize(prep.ctx.device)
                t = time.perf_counter()
                self.phase_s[name] = t - t0
                t0 = t

            multi, ctx = open_gpus(args.numGpus)
            boolean = _bool(args.booleanData)
            users_wanted = _read_ids(args.usersFile) if args.usersFile else None
            items_wanted = _read_ids(args.itemsFile) if args.itemsFile else None
            events = ingest.Events.parse_file(args.input, boolean_data=boolean, ctx=ctx)
            prep = events.prepare(args.minPrefsPerUser)
            events.close()
            phase("prepare")
            lines = []
            if prep.num_items > 0:
                exact = args.similarityClassname in EXACT_MEASURES
                if multi is not None:
                    lists = multi_item_similarity(multi, prep, args, exact)
                elif exact:
                    lists = sim.exact_item_similarity(
                        prep.row, prep.user, prep.pref, prep.num_items, k=args.maxSimilaritiesPerItem,
                        threshold=args.threshold, frac_bits=args.fracBits, precision=args.precision,
                        ucol=prep.ucol, num_users=prep.num_users, device=True)
                else:
                    lists = sim.item_similarity(
                        prep.row, prep.user, prep.pref, prep.num_items, k=args.maxSimilaritiesPerItem,
                        threshold=args.threshold, width=args.sketchWidth, depth=args.sketchDepth,
                        seed=args.sketchSeed, frac_bits=args.fracBits, precision=args.precision, device=True)
                phase("similarity")
                if args.outputPathForSimilarityMatrix:
                    from . import seqfile
                    seqfile.write_similarity_matrix(args.outputPathForSimilarityMatrix,
                                                    *(x.cpu().numpy() if hasattr(x, "cpu") else x for x in lists),
                                                    prep.index_values)
                uv = ib.user_vectors(prep.row, prep.user, prep.pref)
                user_ids = uv.user_ids.cpu().numpy()
                rows = np.arange(user_ids.shape[0], dtype=np.int64)
                if users_wanted is not None:
                    rows = rows[np.isin(user_ids, np.asarray(users_wanted, np.int64))]
                mask = None if items_wanted is None else ib.allowed_mask(prep.item_id, items_wanted)
                if multi is not None:
                    rec = multi.item_based(lists, uv, prep.item_id)
                    phase("replicate")
                    items, vals, cnt = rec.recommend(rows, how_many=args.numRecommendations,
                                                     max_prefs_per_user=args.maxPrefsPerUser, boolean_data=boolean,
                                                     allowed=mask)
                    rec.close()
                else:
                    dev = uv.user_ptr.device
                    allowed = None if mask is None else torch.from_numpy(mask.view(np.int32)).to(dev)
                    item_id = torch.from_numpy(prep.item_id).to(dev)
                    items, vals, cnt = ib.recommend(lists, uv, item_id, torch.from_numpy(rows).to(dev),
                                                    how_many=args.numRecommendations,
                                                    max_prefs_per_user=args.maxPrefsPerUser, boolean_data=boolean,
                                                    allowed=allowed, ctx=prep.ctx)
                    items, vals, cnt = (x.cpu().numpy() for x in (items, vals, cnt))
                phase("recommend")
                for t, r in enumerate(rows):
                    if cnt[t]:
                        lines.append(format_line(user_ids[r], items[t, :cnt[t]], vals[t, :cnt[t]]))
            prep.close()
            with open(args.output, "w") as out:
                out.writelines(lines)
            self.phase_s["write"] = time.perf_counter() - t0
        except Exception as e:   # AbstractJob: failures surface as a non-zero exit code
            print(f"recommenditembased failed: {e}", file=sys.stderr)
            return -1
        finally:
            if multi is not None:
                multi.close()
        return 0


def main(argv=None) -> int:
    return RecommenderJob().run(sys.argv[1:] if argv is None else argv)


if __name__ == "__main__":
    sys.exit(main())
