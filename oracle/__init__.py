"""oracle/ — CPU restatement of the reference's LG-LDM sampling path (TEST INFRASTRUCTURE ONLY).

Nothing here is shipped or measured as the product: only tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py may import this package. The product path
(face-diffusion-model_b200/) never imports it and fails loudly without its CUDA extension.

Parity status: PINNED. Every function below is checked against the reference's own modules
(imported from a reference checkout by oracle/gen_golden.py, with the harness shims of SURVEY.md §8(c));
the resulting vectors are committed under tests/golden/ and re-checked by tests/test_oracle_golden.py.
The HuBERT / wav2vec2 arithmetic lives in the third-party `transformers` package (pinned 4.32.0 by the
reference, 5.5.0 when the vectors were recorded, source not in the reference checkout); the
oracle calls the installed module with shared weights, so parity at that boundary is pinned to the
installed package, not to the reference's pin.
"""
