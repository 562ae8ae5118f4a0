#!/bin/bash
# rebuild libard_b200.so from the repo root (cwd-independent)
cd "$(dirname "$0")/.." && python __graft_entry__.py "$@"
