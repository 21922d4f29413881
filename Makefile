# Convenience targets; everything is also runnable directly (README.md).
PY ?= python

.PHONY: build test test-gpu bench bench-reference reference parity sanitizer golden pin clean

build:            ## nvcc -gencode arch=compute_100a,code=sm_100a -> prysm_b200/_lib/libprysm_b200.so (cross-compiles without a GPU)
	$(PY) prysm_b200/build.py

test: build       ## oracle vs the reference's golden vectors, C ABI, host logic, gloo x 2 (no GPU needed)
	$(PY) -m pytest tests -x -q -m "not gpu"

test-gpu: build   ## parity of the CUDA path through the C ABI (needs a B200)
	$(PY) -m pytest tests -x -q -m gpu

bench: build      ## BASELINE.json metric, one JSON line
	$(PY) bench.py

bench-reference:  ## the reference's algorithm on the host cores, same metric
	$(PY) bench.py --impl reference

reference:        ## install the unmodified reference into oracle/_ref (the --impl reference arm, the drop-in tests)
	bash oracle/install_reference.sh $(PRYSM_REFERENCE)

parity:           ## full-array parity report of C2..C5 against the reference's fp64 run (needs a B200 and oracle/_ref)
	$(PY) tools/parity_report.py

sanitizer:        ## compute-sanitizer memcheck + racecheck over the small-size parity tests (needs a B200)
	bash tools/run_sanitizer.sh

pin:              ## run every oracle function beside the unmodified reference (needs /root/reference)
	PYTHONDONTWRITEBYTECODE=1 $(PY) oracle/check_against_reference.py

golden:           ## regenerate tests/golden/*.npz from the unmodified reference (needs /root/reference)
	PYTHONDONTWRITEBYTECODE=1 $(PY) oracle/make_golden.py

clean:
	rm -rf prysm_b200/_lib .pytest_cache .hypothesis
