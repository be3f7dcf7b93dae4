#!/bin/bash
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 900 python -m pytest -q tests/test_sde.py -m gpu -p no:cacheprovider 2>&1 | tail -3
