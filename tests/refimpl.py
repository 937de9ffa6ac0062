"""
Loader for the UNMODIFIED reference modules (`graphinvent/gnn` of a GraphINVENT checkout), used only by the
fixture generators under `tests/golden/` to pin the oracle.  The checkout is found through the environment variable
GRAPHINVENT_REFERENCE (the repository root of MolecularAI/GraphINVENT); the test-suite itself never imports it.
Recipe = SURVEY.md Appendix C: `gnn/*` imports only torch.
"""
import os
import sys

REPO = os.environ.get("GRAPHINVENT_REFERENCE", "")
REF_ROOT = os.path.join(REPO, "graphinvent")
DATA = os.path.join(REPO, "data")


def available():
    return bool(REPO) and os.path.isdir(os.path.join(REF_ROOT, "gnn"))


def load():
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import gnn.mpnn  # noqa: E402
    return gnn.mpnn


def build(constants):
    m = load()
    cls = {"GGNN": m.GGNN, "MNN": m.MNN, "AttGGNN": m.AttentionGGNN, "EMN": m.EMN}[constants.model]
    return cls(constants)


def read_gdb13_h5(path, n_nodes=13, n_feat=8, n_edge=3, apd=625):
    """Raw-offset reader for the reference's HDF5 fixtures (no h5py here): three
    contiguous int8 datasets after a 2048-byte header, alphabetical order
    APDs / edges / nodes (SURVEY.md §4)."""
    import numpy as np
    raw = np.fromfile(path, np.int8)
    row = apd + n_nodes * n_nodes * n_edge + n_nodes * n_feat
    n = (raw.size - 2048) // row
    o = 2048
    apds = raw[o:o + n * apd].reshape(n, apd); o += n * apd
    edges = raw[o:o + n * n_nodes * n_nodes * n_edge].reshape(n, n_nodes, n_nodes, n_edge)
    o += n * n_nodes * n_nodes * n_edge
    nodes = raw[o:o + n * n_nodes * n_feat].reshape(n, n_nodes, n_feat)
    return nodes, edges, apds
