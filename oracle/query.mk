# Builds the oracle of the volume queries (test infrastructure) as a library of its own, with the flags of Makefile's
# librr_oracle.so:  make -C oracle -f query.mk
CXX      := /usr/bin/g++
CXXFLAGS := -std=c++17 -O2 -fPIC -fopenmp -ffp-contract=off -fno-fast-math -mfma -Wall -Wno-unknown-pragmas

librr_oracle_query.so: ro_query.cpp ro_query.h ro_sample.h ro_math.h
	$(CXX) $(CXXFLAGS) -shared -o $@ ro_query.cpp

clean:
	rm -f librr_oracle_query.so
.PHONY: clean
