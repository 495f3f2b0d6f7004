"""TEST INFRASTRUCTURE ONLY -- never imported by the product package `zstdlite_b200`.

Two CPU checkers live here:
  * `oracle.ref`     ctypes binding of the system's libzstd (libzstd.so.1, 1.5.x), the same
                     library the reference vendors (1.5.6); no sources of it live in this repository.
  * `oracle.restate` ctypes binding of oracle/libzl_oracle.so, our plain-C restatement of the
                     decoder (oracle/zl_oracle.c), pinned against the above and the golden vectors.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs use them.
"""
