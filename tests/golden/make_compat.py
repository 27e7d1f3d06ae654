"""Generate the reference's command-line and data-loader answers by running the UNMODIFIED reference (needs its source tree, oracle/ref_shim.py).

    python tests/golden/make_compat.py

Writes tests/golden/reference_compat.json, read by tests/test_reference_compat.py:
  parser/defaults   vars(parse_args()) of the reference's utility/parser.py with an empty command line
  parser/typical    the same for TYPICAL_ARGV (includes the type=bool quirk of --mask)
  loader/*          what the reference's Data (utility/load_data.py) reads from the seeded tiny dataset of make_golden.py
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, HERE)

TYPICAL_ARGV = ["--dataset", "netflix", "--embed_size", "128", "--weight_size", "[128,128]", "--lr", "0.01", "--mask", "False"]


def _parse(parser_mod, argv):
    saved, sys.argv = sys.argv, ["x"] + list(argv)
    try:
        return vars(parser_mod.parse_args())
    finally:
        sys.argv = saved


def main():
    from llmrec_b200.synth import make_dataset
    from make_golden import TINY, TINY_FLAGS
    from oracle.ref_shim import import_reference

    root = tempfile.mkdtemp(prefix="llmrec_compat_") + "/"
    make_dataset(root, **TINY)
    ref = import_reference(["--data_path", root, "--dataset", "netflix_valid_item"] + TINY_FLAGS)
    parser_mod = sys.modules["utility.parser"]
    d = ref.data_generator
    out = {
        "parser/defaults": _parse(parser_mod, []),
        "parser/typical_argv": TYPICAL_ARGV,
        "parser/typical": _parse(parser_mod, TYPICAL_ARGV),
        "loader/n_users": int(d.n_users), "loader/n_items": int(d.n_items), "loader/n_train": int(d.n_train),
        "loader/exist_users": [int(u) for u in d.exist_users],
        "loader/train_items": {str(u): [int(i) for i in v] for u, v in d.train_items.items()},
        "loader/test_set": {str(u): [int(i) for i in v] for u, v in d.test_set.items()},
        "loader/R_nnz": int(d.R.nnz), "loader/R_shape": list(d.R.shape),
    }
    path = os.path.join(HERE, "reference_compat.json")
    with open(path, "w") as f:
        json.dump(out, f, sort_keys=True)
        f.write("\n")
    print("wrote", path)


if __name__ == "__main__":
    main()
