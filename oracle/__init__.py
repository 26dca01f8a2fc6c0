"""oracle/ — CPU restatement of the reference's algorithm for the LIReC hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under lirec_b200/ may import this package; it is used by
tests/, by __graft_entry__.smoke() and by bench.py's cpu_baseline / --impl reference legs, as
the checker and the reported CPU baseline, never as the product path.

Parity status: the reference ships no tests, golden vectors or fixtures for this path
(SURVEY.md §4, §8c), so the restatement is pinned against the reference ITSELF: the unmodified
reference modules, imported through oracle/reference_shim.py where a reference tree is available,
generated the golden input/output vectors committed under tests/golden/
(tests/golden/make_golden.py), which the restatement is checked against everywhere.
"""
