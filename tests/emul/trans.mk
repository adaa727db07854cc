# Host emulation of the transposed product (test infrastructure; see trans_emul.cpp).
CXX ?= g++
CSRC := ../../sparsex_b200/csrc
libtrans_emul.so: trans_emul.cpp warp_emul.hpp $(CSRC)/part_dev.cuh $(CSRC)/gather_kernel.cuh $(CSRC)/gpu_layout.hpp $(CSRC)/encoder.o $(CSRC)/gpu_layout.o $(CSRC)/mmf.o
	$(CXX) -O1 -g -std=c++17 -fPIC -Wall -Wno-unused-function -pthread -shared -x c++ trans_emul.cpp -x none $(CSRC)/encoder.o $(CSRC)/gpu_layout.o $(CSRC)/mmf.o -o $@
