"""oracle/ -- TEST INFRASTRUCTURE ONLY (not product code).

CPU restatement of the InterDiff sampling hot path (SURVEY.md section 8) used as the
parity checker for the sm_100a CUDA path in interdiff_b200/.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this package.  The product package (interdiff_b200/) never imports it and
fails loudly when its CUDA library is missing.

Pinning status (see DESIGN.md "Oracle"):
  * oracle.restate is checked in tests/test_oracle_vs_reference.py and tests/test_golden.py
    against golden vectors generated from the reference's OWN classes (interdiff/model,
    interdiff/diffusion, interdiff/libsmpl, interdiff/data/tools.py, interdiff/tools.py)
    imported from the reference tree through oracle.shims (oracle/make_golden.py ->
    tests/golden/).
  * Third-party arithmetic whose source is NOT under /root/reference is restated from the
    published algorithm and is "parity unpinned" at that boundary:
      - local_attention.LocalAttention (unpinned version; both rotary placements kept,
        'absolute' is the default, see oracle/local_attention_restated.py)
      - chamfer_distance (first-minimum squared-L2 argmin)
      - pytorch3d.transforms 0.7.2
      - pointnet2_ops 3.0.0 (furthest_point_sampling, ball_query, grouping: oracle/pointnet2_restated.py; the
        golden vector of the point-cloud encoder is the reference's own PointNet2Encoder class running on these
        restated operators)
"""
