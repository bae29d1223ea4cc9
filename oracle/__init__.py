"""CPU oracle for the InvPref hot path.  TEST INFRASTRUCTURE ONLY.

Nothing under ``oracle/`` is part of the product: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import it, and there only as the checker / the timed CPU baseline.
The product path (``invpref_kdd_2022_b200``) never imports this package and fails
loudly when its CUDA extension is missing.

Contents
--------
``invpref_numpy``      closed-form numpy restatement (fp32 or fp64) of the reference's
                       forward / loss / backward / Adam / EM re-assignment, each
                       function citing the reference file:line it follows.
``invpref_torch_cpu``  torch-eager CPU restatement that issues the same ATen op
                       sequence as the reference trainer (autograd + torch.optim.Adam);
                       it is what ``bench.py`` times as the CPU baseline ("port").
``ref_shim``           imports the *live* reference from ``oracle/_ref`` (a checkout of
                       the original project, when present) to pin the two restatements and to
                       generate the golden fixtures under ``tests/golden/``.

Parity pinning: the reference ships no tests and no golden vectors (SURVEY.md §4), so
the oracle is pinned against outputs of the reference itself, run in the build
container by ``tests/golden/make_golden.py`` and committed as ``tests/golden/*.npz``.
"""
