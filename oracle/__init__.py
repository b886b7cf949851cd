"""CPU oracle for the DCLL hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Everything under ``oracle/`` is a CPU restatement (numpy / torch-CPU) of the
reference algorithm for the hot path named in BASELINE.json.  It exists only
so that the CUDA path can be checked against it.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it.  The product package
(``snn_modulation_classification_b200``) never imports this package and has no
CPU fallback.

Pinning: the reference ships no tests and no golden vectors (SURVEY.md section 4),
so the oracle is pinned against outputs of the reference classes themselves,
executed from a checkout of the original project (BASELINE.json's
reference_path, or DCLL_REFERENCE_ROOT) with four import shims
(``oracle/refshim.py``).  The resulting fixtures live in ``tests/golden/`` next
to the script that generated them (``tests/golden/make_golden.py``), and
``tests/test_oracle_vs_reference.py`` re-checks the oracle against the live
reference whenever that checkout or its vendored copy ``oracle/_ref`` is present.

The quantised-weight path has NO counterpart in the reference ("parity
unpinned", SURVEY.md section 8c); ``oracle/quant.py`` is the defining restatement.
"""
