"""Reference arm of bench.py and the drop-in tests: the UNMODIFIED reference, installed under oracle/_ref/
(not under version control) by build().  See oracle/ref_install.py / ref_loader.py."""
