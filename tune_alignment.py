#!/usr/bin/env python
"""Root-level launcher, like infer_ali.py:
    python tune_alignment.py --model <checkpoint> --dataset <name> --scp <list> --output_dir <dir> [--strict]
        [--medfilt_widths 3 5 7] [--aggrs mean topk] [--topks 1 5 10 15 20] [--weights 1,1,0 1,0,0 0,1,0]
The implementation lives in whisper_char_alignment_b200/cli/tune_alignment.py."""
from whisper_char_alignment_b200.cli.tune_alignment import main

if __name__ == "__main__":
    main()
