"""
TEST INFRASTRUCTURE ONLY -- never imported by the product package.

Loads the *unmodified* PhaMers reference modules (scripts/kmer.py, scripts/learning.py,
scripts/phamer.py) under Python 3 so that they can serve as the live oracle in the build
container.  The reference is Python 2.7 and depends on packages that are not installed
here (Bio, matplotlib), so six shims are installed into sys.modules / builtins before
the import (SURVEY.md section 8(c)):

  1. builtins.xrange = range                       (kmer.py:47, phamer.py:251 use xrange)
  2. Bio / Bio.SeqIO with a FASTA ``parse``          (kmer.py:16,135 ; fileIO.py:9)
  3. matplotlib / matplotlib.pyplot stubs           (phamer.py:13-19,32)
  4. sklearn.neighbors.kde -> KernelDensity         (learning.py:15, 2016-era import path)
  5. empty ``basic`` module                         (phamer.py:28 ; basic.py is py2-only syntax)
  6. ``fileIO`` stub with get_fasta_ids/read_fasta  (kmer.py:18,125 ; fileIO.py is py2-only syntax)

The original scripts are found through $PHAMERS_REF (their scripts/ directory); the
repository does not carry them.  This module is used by tests/golden/make_golden.py to
generate the committed golden vectors and, when $PHAMERS_REF is set, by
tests/test_oracle.py to pin oracle/phamers_oracle.py against the real code as well.
"""
import builtins
import importlib
import os
import sys
import types

# the scripts/ directory of an original PhaMers checkout; the repository does not carry one
REF_CANDIDATES = [
    os.environ.get("PHAMERS_REF", ""),
]


def reference_scripts_dir():
    for cand in REF_CANDIDATES:
        if cand and os.path.isfile(os.path.join(cand, "kmer.py")):
            return cand
    return None


def reference_available():
    return reference_scripts_dir() is not None


class _Record(object):
    __slots__ = ("id", "seq", "description")

    def __init__(self, title, seq):
        self.description = title
        self.id = title.split(None, 1)[0] if title.split() else ""
        self.seq = seq


def fasta_parse(handle, fmt="fasta"):
    """Biopython-compatible FASTA tokenisation (SimpleFastaParser semantics): a record
    starts at a line beginning with '>', the id is the first whitespace token of the
    title, the sequence is every following line rstripped, joined, with blanks and CR
    removed."""
    assert fmt == "fasta"
    title, chunks = None, []
    for line in handle:
        if isinstance(line, bytes):
            line = line.decode("ascii", "replace")
        if line.startswith(">"):
            if title is not None:
                yield _Record(title, "".join(chunks).replace(" ", "").replace("\r", ""))
            title, chunks = line[1:].rstrip(), []
        elif title is not None:
            chunks.append(line.rstrip())
    if title is not None:
        yield _Record(title, "".join(chunks).replace(" ", "").replace("\r", ""))


def _install_shims(get_id):
    builtins.xrange = range

    bio = types.ModuleType("Bio")
    seqio = types.ModuleType("Bio.SeqIO")
    seqio.parse = fasta_parse
    bio.SeqIO = seqio
    sys.modules["Bio"] = bio
    sys.modules["Bio.SeqIO"] = seqio

    mpl = types.ModuleType("matplotlib")
    mpl.use = lambda *a, **k: None
    mpl.rcParams = {}
    plt = types.ModuleType("matplotlib.pyplot")
    mpl.pyplot = plt
    sys.modules["matplotlib"] = mpl
    sys.modules["matplotlib.pyplot"] = plt

    import sklearn.neighbors
    kde = types.ModuleType("sklearn.neighbors.kde")
    kde.KernelDensity = sklearn.neighbors.KernelDensity
    sys.modules["sklearn.neighbors.kde"] = kde

    sys.modules["basic"] = types.ModuleType("basic")

    import gzip
    import numpy as np
    fio = types.ModuleType("fileIO")

    def _open(path):
        return gzip.open(path, "rt") if path.endswith(".gz") else open(path, "r")

    def get_fasta_ids(fasta_file):
        with _open(fasta_file) as f:
            return np.array([get_id(str(r.id)) for r in fasta_parse(f)])

    def read_fasta(fasta_file):
        with _open(fasta_file) as f:
            recs = list(fasta_parse(f))
        return np.array([get_id(str(r.id)) for r in recs]), [str(r.seq) for r in recs]

    fio.get_fasta_ids = get_fasta_ids
    fio.read_fasta = read_fasta
    sys.modules["fileIO"] = fio


def _contig_get_id(header):
    # id_parser.get_id for the only header family the synthetic workloads use ('_ID_' contigs,
    # id_parser.py:18-29,95-96); other headers fall back to the first token.
    if "_ID_" in header:
        parts = header.strip().replace(">", "").split("_")
        return parts[1 + parts.index("ID")].replace("-circular", "")
    return header.split(" ")[0]


_cache = {}


def load_reference():
    """Returns (kmer, learning, phamer) reference modules, imported unmodified."""
    if "mods" in _cache:
        return _cache["mods"]
    d = reference_scripts_dir()
    if d is None:
        raise RuntimeError("original PhaMers scripts not found: set PHAMERS_REF to their scripts/ directory")
    _install_shims(_contig_get_id)
    saved = {name: sys.modules.pop(name, None) for name in ("kmer", "learning", "phamer")}
    sys.path.insert(0, d)
    try:
        kmer = importlib.import_module("kmer")
        learning = importlib.import_module("learning")
        phamer = importlib.import_module("phamer")
    finally:
        sys.path.remove(d)
    # keep them out of sys.modules under the bare names so they can never shadow the
    # product's own phamers_b200.kmer / phamers_b200.phamer
    for name in ("kmer", "learning", "phamer"):
        mod = sys.modules.pop(name)
        sys.modules["_phamers_reference_" + name] = mod
        if saved[name] is not None:
            sys.modules[name] = saved[name]
    import logging
    for m in (kmer, learning, phamer):
        m.logger.setLevel(logging.ERROR)
    _cache["mods"] = (kmer, learning, phamer)
    return _cache["mods"]


def load_reference_cross_validate():
    """The unmodified scripts/cross_validate.py, imported against the reference kmer / learning / phamer modules."""
    if "cv" in _cache:
        return _cache["cv"]
    kmer, learning, phamer = load_reference()
    d = reference_scripts_dir()
    names = {"kmer": kmer, "learning": learning, "phamer": phamer}
    saved = {name: sys.modules.get(name) for name in list(names) + ["cross_validate"]}
    sys.modules.update(names)
    sys.path.insert(0, d)
    try:
        sys.modules.pop("cross_validate", None)
        cv = importlib.import_module("cross_validate")
    finally:
        sys.path.remove(d)
        for name, mod in saved.items():
            if mod is None:
                sys.modules.pop(name, None)
            else:
                sys.modules[name] = mod
    import logging
    cv.logger.setLevel(logging.ERROR)
    _cache["cv"] = cv
    return cv
