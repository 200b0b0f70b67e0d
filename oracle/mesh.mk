# Builds the oracle of the surface extraction (test infrastructure) as a library of its own, with the flags of Makefile's
# librr_oracle.so:  make -C oracle -f mesh.mk
CXX      := /usr/bin/g++
CXXFLAGS := -std=c++17 -O2 -fPIC -fopenmp -ffp-contract=off -fno-fast-math -mfma -Wall -Wno-unknown-pragmas

librr_oracle_mesh.so: ro_mesh.cpp ro_mesh.h ro_sample.h ro_math.h
	$(CXX) $(CXXFLAGS) -shared -o $@ ro_mesh.cpp

clean:
	rm -f librr_oracle_mesh.so
.PHONY: clean
