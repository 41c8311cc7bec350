"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the PhotoVerse dual-branch conditioning hot path.

This package restates, in plain PyTorch CPU arithmetic (fp32 / fp64), what the reference
computes in

  * models/attention_processor.py:245-435  (PhotoVerseAttnProcessor2_0.__call__)
  * models/attention_processor.py:27-56    (constructor validation / parameters)
  * models/adapters.py:5-44                (PhotoVerseAdapter)
  * models/unet.py:38-47                   (regulariser gather)
  * peft 0.10.0 lora.Linear.forward        (un-vendored dependency, restated from its
                                            published algorithm: y = W x + (alpha/r) B A dropout(x))

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs may import it.  The product package ``photoverse_b200`` never imports ``oracle``.

Pinning: the reference ships NO tests, golden vectors or fixtures for this path (SURVEY.md §4).
The oracle is therefore pinned against the *reference implementation itself*, imported verbatim
from the upstream checkout named by PHOTOVERSE_REFERENCE_ROOT by ``oracle/ref_loader.py`` and compared in
``oracle/make_golden.py`` (which also writes ``tests/golden/*.npz``; re-run it to regenerate).
``tests/test_oracle_golden.py`` re-checks the oracle against those committed outputs everywhere
and against the live reference when PHOTOVERSE_REFERENCE_ROOT is set.
"""
