#! /usr/bin/env python
"""Same name and command line as scripts/select_db.py of the reference; runs metalign_b200.select_db."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from metalign_b200.select_db import select_main, select_parseargs  # noqa: E402

if __name__ == "__main__":
    select_main(select_parseargs(), leave_open=True)      # device memory goes back with the process
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)                      # skip the interpreter's and the CUDA runtime's orderly teardown of GBs of device memory
