# CPU ORACLE of the relative poses (test infrastructure): its own library, so the main oracle build stays as it is.
#   make -C oracle -f relpose.mk
# Same flags as Makefile (-ffp-contract=off, no -ffast-math).  The AC-RANSAC / 5-point sources are compiled in again;
# -Bsymbolic keeps this library's calls inside it when liboracle.so is loaded in the same process.
CXX := g++
CXXFLAGS ?= -O3 -std=c++17 -fPIC -fopenmp -ffp-contract=off -fno-fast-math -Wall -Wextra
SRCS := oracle_relpose.cpp oracle_acransac.cpp oracle_fivepoint.cpp
OUT := _build/liboracle_relpose.so

all: $(OUT)

$(OUT): $(SRCS) oracle.h oracle_relpose.h oracle_detmath.hpp
	mkdir -p _build
	$(CXX) $(CXXFLAGS) -shared -Wl,-Bsymbolic -o $@ $(SRCS)

.PHONY: all
