# The host emulation with the bits observation format and level sets (CPU test-suite only; see pgtg_emu_bits.cpp): make -f bits.mk
CXX ?= g++
CXXFLAGS ?= -O1 -g -fPIC -std=c++17 -ffp-contract=off -Wall -Wno-unused-function -Wno-unused-variable -Wno-unknown-pragmas
SRC = ../../pgtg_b200/csrc
DEPS = pgtg_emu_bits.cpp pgtg_emu_levels.cpp pgtg_emu.cpp $(SRC)/pgtg_device.cuh $(SRC)/pgtg_logic.cuh $(SRC)/pgtg_phases.cuh $(SRC)/pgtg_traffic.cuh $(SRC)/pgtg_api_impl.hpp $(SRC)/pgtg_env.hpp $(SRC)/pgtg_tables.h ../../include/pgtg_b200.h
all: libpgtg_emu_bits.so
libpgtg_emu_bits.so: $(DEPS)
	$(CXX) $(CXXFLAGS) -x c++ -shared -o $@ pgtg_emu_bits.cpp -lm -lpthread
clean:
	rm -f libpgtg_emu_bits.so
