#! /usr/bin/env python
"""select_db.py for every sample of a sample sheet against one database: one CUDA context and one loaded database per GPU.

    select_many.py samples.tsv data/ [--out_dir DIR] [select_db.py flags that are not tied to one sample]

Each sample's files go to DIR/<sample_id>/, and DIR/samples_summary.tsv lists every sample's status.  The exit status is 1
when any sample failed.  Under torchrun the samples are spread over the GPUs of the node (metalign_b200.select_db.select_many)."""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from metalign_b200.select_db import SUMMARY_NAME, select_many, select_many_parseargs  # noqa: E402

if __name__ == "__main__":
    args = select_many_parseargs()
    try:
        results = select_many(args.sample_sheet, args)
    except ValueError as e:           # the sheet or --cutoff, refused before any GPU work
        sys.exit("select_many: %s" % e)
    failed = [r for r in results if r.status != "ok"]
    if "torch.distributed" in sys.modules:
        import torch.distributed as tdist
        if tdist.is_initialized():
            tdist.destroy_process_group()
    if failed and int(os.environ.get("RANK", "0")) == 0:
        sys.stderr.write("select_many: %d of %d samples failed (see %s)\n"
                         % (len(failed), len(results), os.path.join(args.out_dir, SUMMARY_NAME)))
    sys.exit(1 if failed else 0)
