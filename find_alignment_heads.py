#!/usr/bin/env python
"""Root-level launcher, like infer_ali.py:
    python find_alignment_heads.py --model <checkpoint> --dataset <name> --scp <list> --output_dir <dir> [--strict]
The implementation lives in whisper_char_alignment_b200/cli/find_alignment_heads.py."""
from whisper_char_alignment_b200.cli.find_alignment_heads import main

if __name__ == "__main__":
    main()
