"""`mahout itemsimilarity` with the GPU sketch-cosine measure -- the job-level drop-in.

    python -m mahout_b200.itemsimilarity --input prefs.csv --output out.tsv \
        --similarityClassname SIMILARITY_COSINE | SIMILARITY_SKETCH_COSINE --maxSimilaritiesPerItem 100 \
        [--minPrefsPerUser 1] [--booleanData true] [--threshold 0.1] \
        [--sketchWidth 4096] [--sketchDepth 4] [--sketchSeed 42] [--precision rescored|tensor] [--numGpus N]

Same flags, input format (`userID,itemID[,pref]`, split on tab or comma) and output format
(`itemA<TAB>itemB<TAB>similarity`, itemA < itemB, ordered by (itemA, itemB)) as the reference's
ItemSimilarityJob (cf/taste/hadoop/similarity/item/ItemSimilarityJob.java:97-232); phase 1
(RowSimilarityJob) is replaced by the native call sequence.  Returns 0 on success, -1 on bad
arguments or failure, like AbstractJob.  SIMILARITY_COSINE is the reference's exact cosine (every
user owns a counter column); SIMILARITY_SKETCH_COSINE the count-min sketch measure of the fork.
`--maxPrefs` is accepted for compatibility: no down-sampling takes place (the dense tensor-core
contraction does not need it), i.e. the job behaves like the reference with --maxPrefs >= every count.
`--numGpus N` (0 = every visible GPU) runs the preparation on the first of N GPUs of this process and phase 1 as one
mb200_job_item_similarity call over all N, as the native driver's flag of the same name does.
"""
from __future__ import annotations

import argparse
import sys

from . import ingest
from . import similarity as sim

# -s SIMILARITY_COSINE (or the measure's class name) is the reference's exact cosine; the sketch measure
# of the fork is selected by its own names
EXACT_MEASURES = ("SIMILARITY_COSINE",
                  "org.apache.mahout.math.hadoop.similarity.cooccurrence.measures.CosineSimilarity")
SKETCH_MEASURES = ("SIMILARITY_SKETCH_COSINE",
                   "org.apache.mahout.math.hadoop.similarity.cooccurrence.measures.NativeSketchCosineSimilarity")
MEASURES = EXACT_MEASURES + SKETCH_MEASURES


def _bool(s: str) -> bool:
    return str(s).strip().lower() == "true"        # Boolean.valueOf


def build_parser() -> argparse.ArgumentParser:
    ap = argparse.ArgumentParser(prog="itemsimilarity", add_help=True)
    ap.add_argument("--input", "-i", required=True)
    ap.add_argument("--output", "-o", required=True)
    ap.add_argument("--similarityClassname", "-s", required=True)
    ap.add_argument("--maxSimilaritiesPerItem", "-m", type=int, default=sim.DEFAULT_MAX_SIMILAR_ITEMS_PER_ITEM)
    ap.add_argument("--maxPrefs", "-mppu", type=int, default=500)
    ap.add_argument("--minPrefsPerUser", "-mp", type=int, default=sim.DEFAULT_MIN_PREFS_PER_USER)
    ap.add_argument("--booleanData", "-b", default="false")
    ap.add_argument("--threshold", "-tr", type=float, default=None)
    ap.add_argument("--randomSeed", type=int, default=None)
    ap.add_argument("--tempDir", default=None)
    ap.add_argument("--startPhase", type=int, default=0)
    ap.add_argument("--endPhase", type=int, default=2 ** 31 - 1)
    ap.add_argument("--sketchWidth", type=int, default=4096)
    ap.add_argument("--sketchDepth", type=int, default=4)
    ap.add_argument("--sketchSeed", type=int, default=42)
    ap.add_argument("--fracBits", type=int, default=1)
    ap.add_argument("--precision", default="rescored", choices=["rescored", "certified", "tensor"])
    ap.add_argument("--similarityMatrixOutput", default=None,
                    help="also write phase 1's output: SequenceFile<IntWritable,VectorWritable> rows of the "
                         "similarity matrix (what RecommenderJob / phase 2 read)")
    ap.add_argument("--numGpus", type=int, default=None,
                    help="run phase 1 on N GPUs of this process (0 = every visible GPU)")
    return ap


def open_gpus(num_gpus):
    """(MultiGpu, the Context of its first GPU) for --numGpus N, (None, None) without the flag"""
    if num_gpus is None:
        return None, None
    from .multi import MultiGpu
    multi = MultiGpu(num_gpus)
    return multi, multi.context(0)


def multi_item_similarity(multi, prep, args, exact: bool):
    """phase 1 over every GPU of `multi` from prepared prefs: the host columns go to mb200_job_item_similarity; the
    exact measure as a depth-1 bank of one column per user (hash a = 1, b = 0), as the native driver passes it.
    Returns numpy (idx [I, k], sim [I, k], cnt [I])."""
    row, pref = prep.row.cpu().numpy(), prep.pref.cpu().numpy()
    if exact:
        key, width, depth, hp = prep.ucol.cpu().numpy(), max(prep.num_users, 1), 1, ([1], [0])
    else:
        key, width, depth, hp = prep.user.cpu().numpy(), args.sketchWidth, args.sketchDepth, None
    idx, s, cnt, _ = multi.item_similarity(row, key, pref, prep.num_items, k=args.maxSimilaritiesPerItem,
                                           threshold=args.threshold, width=width, depth=depth, seed=args.sketchSeed,
                                           frac_bits=args.fracBits, precision=args.precision, hash_params=hp)
    return idx, s, cnt


class ItemSimilarityJob:
    def run(self, argv) -> int:
        try:
            args = build_parser().parse_args(argv)
        except SystemExit:
            return -1
        if args.similarityClassname not in MEASURES:
            print(f"itemsimilarity: the native path implements the cosine measure only "
                  f"(got {args.similarityClassname})", file=sys.stderr)
            return -1
        if args.maxSimilaritiesPerItem <= 0:
            print("maxSimilarItemsPerItem must be greater then 0!", file=sys.stderr)
            return -1
        multi = None
        try:
            multi, ctx = open_gpus(args.numGpus)
            # PreparePreferenceMatrixJob on the GPU: the text goes to the device once, the events stay there
            events = ingest.Events.parse_file(args.input, boolean_data=_bool(args.booleanData), ctx=ctx)
            prep = events.prepare(args.minPrefsPerUser)
            events.close()
            if prep.num_items == 0:
                idx = s = cnt = ()
                pairs = []
            else:
                if multi is not None:
                    idx, s, cnt = multi_item_similarity(multi, prep, args, args.similarityClassname in EXACT_MEASURES)
                elif args.similarityClassname in EXACT_MEASURES:
                    idx, s, cnt = sim.exact_item_similarity(
                        prep.row, prep.user, prep.pref, prep.num_items, k=args.maxSimilaritiesPerItem,
                        threshold=args.threshold, frac_bits=args.fracBits, precision=args.precision,
                        ucol=prep.ucol, num_users=prep.num_users)
                else:
                    idx, s, cnt = sim.item_similarity(
                        prep.row, prep.user, prep.pref, prep.num_items, k=args.maxSimilaritiesPerItem,
                        threshold=args.threshold, width=args.sketchWidth, depth=args.sketchDepth,
                        seed=args.sketchSeed, frac_bits=args.fracBits, precision=args.precision)
                pairs = sim.most_similar_item_pairs(idx, s, cnt, prep.item_id)
                if args.similarityMatrixOutput:
                    from . import seqfile
                    seqfile.write_similarity_matrix(args.similarityMatrixOutput, idx, s, cnt, prep.index_values)
            prep.close()
            with open(args.output, "w") as out:
                for a, b, v in pairs:
                    out.write(f"{a}\t{b}\t{sim.java_double_to_string(v)}\n")
        except Exception as e:   # AbstractJob: failures surface as a non-zero exit code
            print(f"itemsimilarity failed: {e}", file=sys.stderr)
            return -1
        finally:
            if multi is not None:
                multi.close()
        return 0


def main(argv=None) -> int:
    return ItemSimilarityJob().run(sys.argv[1:] if argv is None else argv)


if __name__ == "__main__":
    sys.exit(main())
