"""
CPU oracle for the foldingdiff reverse-diffusion sampler.

THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference``
legs of ``bench.py`` may import anything from this package, and only as the
checker or as the timed CPU baseline - never as a fallback for the CUDA path.

Parity status: **parity unpinned at the HuggingFace boundary.**  The encoder
arithmetic of the reference lives in ``transformers==4.11.3`` (pinned in
/root/reference/environment.yml:14, requirements.txt:6), which is not
installable in this image (transformers 5.5.0 has no ``relative_key`` code).
``oracle/forward.py`` restates that published algorithm; no reference test
pins encoder *values*.  The restated layer IS cross-checked against HF's own
code in the installed transformers (``tests/test_oracle_hf_crosscheck.py``:
``Wav2Vec2BertSelfAttention`` with ``relative_key`` + ``BertSelfOutput`` /
``BertIntermediate`` / ``BertOutput`` on the real fixture weights, 7e-7), which
leaves only the sign convention of the distance index (l - r) resting on the
4.11.3 source text.  Everything around the encoder IS pinned: the loop,
schedules, noise sampling and wrap are checked against the reference's own
code (imported from /root/reference under ``oracle/ref_shims.py`` in the
authoring container; outputs committed as ``tests/golden/*.npz`` together with
``tests/golden/make_golden.py``), and against the known answers recorded in
SURVEY.md Appendix A.3/A.4.

Modules
-------
forward.py    restated noise-predictor forward (modelling.py:384-484 + HF 4.11.3 encoder)
schedules.py  beta schedules / alpha tables (beta_schedules.py:20-78)
loop.py       p_sample / p_sample_loop / sample_noise / wrap (sampling.py:27-132,
              datasets.py:772-799, utils.py:87-121)
nerf.py       NeRF backbone builder (nerf.py:79-204), bit-identical to the reference module
writers.py    csv.gz (= the reference's own DataFrame.to_csv call) and PDB text (pinned on a reference-written file)
loss.py       the training objective (losses.py:12-62, modelling.py:553-604, :684-685) and its gradient in closed form:
              groundwork for SURVEY 8f rank 3, no CUDA counterpart yet; bit-identical to the reference's functions
replay.py     digests and model-call record / replay for comparing with the reference's stored answers
ref_shims.py  sys.modules stubs that make the reference's own loop importable
              (authoring container only; /root/reference does not exist on the GPU box)
"""
