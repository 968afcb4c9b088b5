"""Command-line drivers (ports of the reference's mbd/scripts)."""
