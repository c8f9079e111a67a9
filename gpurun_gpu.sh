python -c "import __graft_entry__ as g; g.build()" || exit 1
timeout 1500 python -m pytest tests/test_kernel_units.py -m gpu -q -s -rxXs -p no:cacheprovider 2>&1 | grep -E "^\[gpu\] flank|passed|failed|FAILED|^E " | cut -c1-900
