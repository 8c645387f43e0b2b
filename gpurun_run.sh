python -c "import __graft_entry__ as g; g.build()" > /dev/null 2>&1 || exit 1
timeout 480 python -m pytest tests -m gpu -q -p no:cacheprovider 2>&1 | tail -6
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
