"""Alignment ingest (SURVEY 8f N3; reference src/msa.cpp:18-88: PHYLIP interleaved, then PHYLIP
sequential, then FASTA) -- the same alignment in every on-disk form gives the same model: the same
compressed site patterns and the same log-likelihood bits (oracle backend).  Ragged, empty and
inconsistent inputs are refused the way the reference refuses them."""
import textwrap

import numpy as np
import pytest

import fixtures
import oracle_build
import oracle_capi
from root_digger_b200 import capi


@pytest.fixture(scope="module")
def lib():
    oracle_capi.load_oracle().rdo_set_default_mode(oracle_capi.MODE_ENGINE)
    return capi.load_tree_lib(oracle_build.build_host_on_oracle())


@pytest.fixture(scope="module")
def case():
    fx = fixtures.load("10.fasta")
    labels = list(fx["alignment"])
    seqs = [fx["alignment"][l] if isinstance(fx["alignment"][l], str) else fx["alignment"][l].decode() for l in labels]
    return fx, labels, seqs


def writers():
    def phylip_one_line(labels, seqs):
        return "%d %d\n" % (len(labels), len(seqs[0])) + "".join("%s %s\n" % (l, s) for l, s in zip(labels, seqs))

    def phylip_sequential_wrapped(labels, seqs):
        out = [" %d   %d" % (len(labels), len(seqs[0]))]
        for l, s in zip(labels, seqs):
            out.append(l)
            out += textwrap.wrap(s, 70)
        return "\n".join(out) + "\n"

    def phylip_interleaved(labels, seqs, block=60):
        out = ["%d %d" % (len(labels), len(seqs[0]))]
        for b in range(0, len(seqs[0]), block):
            for l, s in zip(labels, seqs):
                chunk = " ".join(textwrap.wrap(s[b:b + block], 10))
                out.append(("%-12s%s" % (l, chunk)) if b == 0 else chunk)
            out.append("")
        return "\n".join(out)

    def fasta_wrapped(labels, seqs):
        return "".join(">%s\n%s\n" % (l, "\n".join(textwrap.wrap(s, 50))) for l, s in zip(labels, seqs))

    def fasta_crlf_lowercase(labels, seqs):
        return "".join(">%s \r\n%s\r\n" % (l, s.lower()) for l, s in zip(labels, seqs))

    return dict(phylip_one_line=phylip_one_line, phylip_sequential_wrapped=phylip_sequential_wrapped,
                phylip_interleaved=phylip_interleaved, fasta_wrapped=fasta_wrapped,
                fasta_crlf_lowercase=fasta_crlf_lowercase)


def model_from(lib, fx, path, K=2):
    m = capi.Model.from_files(capi.RootedTree(path=str(fx["tree_path"]), lib=lib), path, None, K, seed=5)
    m.initialize_partitions(uniform_freqs=False)
    return m


def test_every_on_disk_form_gives_the_same_model(lib, case, tmp_path):
    fx, labels, seqs = case
    want = None
    for name, write in writers().items():
        path = tmp_path / (name + ".aln")
        path.write_text(write(labels, seqs), newline="")
        m = model_from(lib, fx, path)
        got = (m.sites(), [m.compute_lh(r).hex() for r in (0, 3, 9)], m.sweep_root_lh().tobytes())
        m.close()
        if want is None:
            want = got
            assert got[0] == 991  # the reference's pattern count for 10.fasta (SURVEY section 4)
        assert got == want, name


def test_row_order_does_not_matter(lib, case, tmp_path):
    """rows are matched to tips by label (src/model.cpp:302-325), not by position"""
    fx, labels, seqs = case
    a, b = tmp_path / "a.fasta", tmp_path / "b.fasta"
    a.write_text("".join(">%s\n%s\n" % p for p in zip(labels, seqs)))
    b.write_text("".join(">%s\n%s\n" % p for p in reversed(list(zip(labels, seqs)))))
    ma, mb = model_from(lib, fx, a), model_from(lib, fx, b)
    # pattern compression orders the columns by content read row by row, so the two models hold
    # the same patterns in (possibly) another order: the log-likelihood agrees to rounding
    assert ma.sites() == mb.sites()
    assert abs(ma.compute_lh(2) - mb.compute_lh(2)) <= 1e-9 * abs(ma.compute_lh(2))
    ma.close()
    mb.close()


@pytest.mark.parametrize("text,why", [
    ("", "empty file"),
    ("\n\n", "blank file"),
    ("2 4\nA ACGT\nB ACG\n", "PHYLIP row shorter than declared, and not a FASTA either"),
    (">A\nACGT\n>B\nACG\n", "ragged FASTA"),
    ("ACGT\n>A\nACGT\n", "FASTA sequence before the first header"),
])
def test_unreadable_alignments_are_refused(lib, case, tmp_path, text, why):
    fx = case[0]
    path = tmp_path / "bad.aln"
    path.write_text(text)
    with pytest.raises(RuntimeError, match="parse msa|match in size|Taxa|could not be created"):
        capi.Model.from_files(capi.RootedTree(path=str(fx["tree_path"]), lib=lib), path, None, 1)


def test_alignment_and_tree_must_name_the_same_taxa(lib, case, tmp_path):
    fx, labels, seqs = case
    missing = tmp_path / "missing.fasta"
    missing.write_text("".join(">%s\n%s\n" % p for p in list(zip(labels, seqs))[:-1]))
    renamed = tmp_path / "renamed.fasta"
    renamed.write_text("".join(">%s\n%s\n" % p for p in zip(labels[:-1] + ["nobody"], seqs)))
    for path in (missing, renamed):
        with pytest.raises(RuntimeError, match="inconsistient|Taxa"):
            capi.Model.from_files(capi.RootedTree(path=str(fx["tree_path"]), lib=lib), path, None, 1)


def test_ambiguity_codes_and_gaps(lib, case, tmp_path):
    """IUPAC unions and gaps are states 1..15 (corax_map_nt); an unknown character is refused when the
    tips are set (src/model.cpp:310-318)"""
    fx, labels, seqs = case
    edited = [s[:5] + "RYKMSWBDHVN-?" + s[18:] for s in seqs]
    ok = tmp_path / "iupac.fasta"
    ok.write_text("".join(">%s\n%s\n" % p for p in zip(labels, edited)))
    m = model_from(lib, fx, ok)
    assert np.isfinite(m.compute_lh(0))
    m.close()
    bad = tmp_path / "bad_char.fasta"
    bad.write_text("".join(">%s\n%s\n" % p for p in zip(labels, [s[:7] + "J" + s[8:] for s in seqs])))
    with pytest.raises(RuntimeError, match="tip|state|character"):
        model_from(lib, fx, bad)


def test_the_reference_sources_read_every_form_through_the_compat_header(lib, case, tmp_path):
    """RootDigger's own src/msa.cpp, compiled unchanged against root_digger_b200/compat/corax/corax.h,
    reads each form through the compat readers (corax_phylip_parse_interleaved / _sequential,
    corax_fasta_getnext in compat/corax_compat.cpp) and its model_t gives, for every root, the bits
    this repository's host gives for the same file.  Compared with the recorded results instead (no
    checkout), neither msa.cpp nor the compat readers run: every form read by this host must then give
    the reference's record of the fixture file."""
    from test_reference_sources import reference
    ref = reference("oracle")  # RootDigger's sources, else their recorded results (reported as a warning)
    fx, labels, seqs = case
    for name, write in writers().items():
        path = tmp_path / (name + ".aln")
        path.write_text(write(labels, seqs), newline="")
        theirs = ref.all_root_lh("10.fasta", 2, 5, alignment=path)
        m = model_from(lib, fx, path)
        ours = m.compute_all_root_lh()
        m.close()
        assert np.array_equal(theirs.view(np.uint64), np.asarray(ours).view(np.uint64)), name
