"""CPU oracle for the colour-modem hot path — TEST INFRASTRUCTURE ONLY.

This package is a float64 numpy/scipy restatement of the reference's per-line
modem chain (kFYatek/color_modem, ``color_modem/*.py``), rewritten as
*stateless, frame-level* functions vectorised over scan lines.  Every function
cites the reference ``file:line`` it follows.

Rules (see DESIGN.md):
  * only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
    ``--impl reference`` legs of ``bench.py`` may import this package;
  * the product (``color_modem_b200``) never imports it and has no CPU fallback.

Parity pin: the reference ships no tests or golden vectors, so the oracle is
pinned against *outputs of the reference itself*: ``tests/golden/make_golden.py``
imports a checkout of the reference named by ``COLOR_MODEM_REFERENCE`` (with the
scipy ``iirdesign`` validation shim described in SURVEY.md §8c), runs
``ImageModem.modulate/demodulate`` for every supported composition/preset and
commits the u8 frames plus a few float64 lines under ``tests/golden/``.
``tests/test_oracle_golden.py`` checks this oracle against those fixtures
(CPU-only), and ``tests/test_oracle_vs_reference.py`` re-checks live whenever
``COLOR_MODEM_REFERENCE`` is set.

Third-party arithmetic: the reference calls ``scipy.signal`` (``lfilter``,
``resample_poly``, ``iirdesign``, ``iirfilter``, ``group_delay``, ``freqz``;
scipy is not pinned by the reference — 1.18.1 here).  Filter *design* is done
with the same scipy calls; ``oracle.dsp`` additionally restates ``lfilter``
(direct-form II transposed) and ``upfirdn``/``resample_poly`` in plain numpy so
the recursion and the polyphase centring arithmetic that the CUDA kernels
implement are written down and checked against scipy.
"""
from .raster import Raster, STANDARDS          # noqa: F401
from .modems import ModemSpec, build            # noqa: F401
from .frame import encode_frame_u8, decode_frame_u8, composite_level, composite_unlevel, to_u8  # noqa: F401
