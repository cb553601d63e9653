"""CPU oracle for the OverlapNet inference hot path.

TEST INFRASTRUCTURE ONLY.  Nothing in ``overlapnet_b200/`` imports this package;
only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import it, and there only as the checker / CPU baseline.

Contents
--------
projection.py  NumPy restatement of ``src/utils/utils.py:59-186`` (range_projection,
               gen_normal_map) and the cue drivers ``src/utils/gen_*_data.py``.
               PARITY PINNED: bit-exact against the reference's shipped fixtures
               (``data/scans/*.bin`` -> ``data/preprocess_data_demo/**.npy``) and against the
               outputs of the reference's own functions stored under tests/golden/
               (tests/test_oracle_*.py, tools/make_golden.py, tools/make_golden_reference.py).
network.py     torch-CPU restatement of the leg (``generateNet.py:119-219``), the delta head
               (``generateNet.py:15-116``), the circular padding (``RangePadding2D.py:31-41``),
               the correlation head (``NormalizedCorrelation2D.py:43-109``) and the readout
               (``infer.py:157-158``).  PARITY UNPINNED by the reference: TensorFlow/Keras/h5py
               are not installable offline and ``data/model_geo.weight`` is not shipped, so no
               reference activation exists to compare with.  It is pinned only by the
               reference's own known-answer statements (RangePadding2D.py:5 KAT, the analytic
               shift KAT of the correlation head) and by an independent naive loop restatement.
gt.py          NumPy restatement of the ground-truth generator ``src/utils/com_overlap_yaw.py:10-68``
               (float64 range projection, float32 image compare, yaw bin).  PARITY PINNED: bit-exact
               against the reference's own ``com_overlap_yaw`` run in the build container
               (tools/make_golden_gt.py -> tests/golden/gt_overlap_yaw.npz).
infer_ref.py   restatement of the ``Infer`` class call semantics (``infer.py:22-265``) on top of
               projection.py + network.py.
"""
