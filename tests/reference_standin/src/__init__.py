"""Stand-in of a checkout of the reference: the package layout install() patches (see tests/test_install.py)."""
