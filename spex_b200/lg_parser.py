"""Command-line surface of the LightGCN_SPEX entry points.

The flag NAMES, types and defaults are the contract (the model and the loaders read
``args.recdim / layer / keepprob / A_split / dropout / a_fold / dataset ...``); they are those of
/root/reference/LightGCN_SPEX/code/lg_parser.py:3-24.  Differences: ``--data_path`` is honoured by
``Loader`` (the reference parses it but hard-codes "../data/", dataloader.py:74) and ``parse_args_r``
accepts an explicit argv for tests.
"""
import argparse

# (flag, type or None for a switch, default, what it controls here)
_FLAGS = (
    ("cuda_id", str, "0", "CUDA_VISIBLE_DEVICES for the run"),
    ("data_path", str, "../data/", "directory that holds <dataset>/rec/*.rating|negative"),
    ("dataset", str, "twitter", "epinion2 | weibo | twitter (directory name under data_path)"),
    ("nb_heads", int, 3, "attention heads of the path-prediction task (main_11)"),
    ("recdim", int, 64, "embedding width D (the sm_100a fast paths are built for 32/64/128)"),
    ("layer", int, 3, "propagation depth K of computer()"),
    ("lr", float, 0.001, "Adam step size"),
    ("dropout", int, 0, "1 = reference RNG stream, 2 = counter-based mask generated on the GPU"),
    ("keepprob", float, 0.6, "probability that an edge survives the dropout"),
    ("a_fold", int, 100, "row folds of the adjacency when A_split is on"),
    ("epochs", int, 50, "training epochs"),
    ("seed", int, 2020, "seed of every generator"),
    ("A_split", int, 0, "1 = getSparseGraph() returns a_fold row blocks"),
    ("batch_size", int, 256, "(kept for compatibility; the rec loader uses 256)"),
    ("batchSize", int, 256, "paths per batch of the path-prediction task"),
    ("hiddenSize", int, 64, "hidden width of the path-prediction task"),
    ("nonhybrid", None, False, "path task: global preference only"),
    ("act", int, 1, "activation selector of the path task"),
)


def build_parser() -> argparse.ArgumentParser:
    parser = argparse.ArgumentParser(description="LightGCN_SPEX on spex_b200")
    for name, kind, default, doc in _FLAGS:
        if kind is None:
            parser.add_argument("--" + name, action="store_true", help=doc)
        elif name == "data_path":
            parser.add_argument("--" + name, nargs="?", default=default, help=doc)
        else:
            parser.add_argument("--" + name, type=kind, default=default, help=doc)
    return parser


def parse_args_r(argv=None):
    return build_parser().parse_args(argv)
