"""Build recipe of the C restatement (oracle/pf_oracle.c -> oracle/libpf_oracle.so).  The reference is pure Python: its
install into oracle/_ref is oracle/reference.py."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle.c_oracle import build  # noqa: E402

if __name__ == "__main__":
    print(build(force=True))
