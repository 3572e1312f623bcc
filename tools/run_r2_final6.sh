python -m pytest tests/ -m gpu -q 2>&1 | tail -4
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
python tools/bench_leaf.py 2>&1 | grep -E "rc=|us per leaf" | tail -3
