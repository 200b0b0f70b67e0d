# Builds the oracle of the point-cloud export (test infrastructure) as a library of its own, with the flags of Makefile's
# librr_oracle.so:  make -C oracle -f cloud.mk
CXX      := /usr/bin/g++
CXXFLAGS := -std=c++17 -O2 -fPIC -fopenmp -ffp-contract=off -fno-fast-math -mfma -Wall -Wno-unknown-pragmas

librr_oracle_cloud.so: ro_cloud.cpp ro_cloud.h ro_draw.h ro_math.h
	$(CXX) $(CXXFLAGS) -shared -o $@ ro_cloud.cpp

clean:
	rm -f librr_oracle_cloud.so
.PHONY: clean
