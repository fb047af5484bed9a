"""oracle/ — TEST INFRASTRUCTURE ONLY (never imported by videollama2_b200).

CPU checkers for the VideoLLaMA2 video->text prefill path:
  * ref_loader.py  imports the UNMODIFIED reference classes from /root/reference (three shims, see SURVEY.md §8c);
                   only usable in the build container (the GPU box has no /root/reference).
  * torch_ref.py   a plain-PyTorch CPU restatement of the same algorithm (each function cites the reference lines);
                   travels to the GPU box; pinned against the real reference by tests/test_oracle_vs_reference.py here
                   and against the committed fixtures in tests/golden/ everywhere.
  * synth.py       configs + deterministic synthetic weights (HF state-dict names) and inputs.
  * make_golden.py regenerates tests/golden/*.pt from the real reference; make_golden_calls.py records the reference
                   calls that tests compare with one by one (tests/golden/reference_calls.pt).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this package.
Parity status: the reference ships no tests or golden vectors for this path (SURVEY.md §4), so the pin is
"outputs of the reference itself run here" (make_golden.py), not reference-provided known answers.
"""
