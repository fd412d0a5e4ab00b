# spf_b200 native build.  `make` builds everything in-tree:
#   spf_b200/libspf_b200.so      the product: sm_100a kernels + C ABI (include/spf_b200.h)
#   spf_b200/csrc/libspf_emu.so  host emulator of the kernel bodies (test infrastructure)
#   oracle/libspf_oracle.so      CPU oracle (test infrastructure)
NVCC ?= nvcc
CXX ?= g++
NVFLAGS ?= -std=c++17 -O3 -fmad=false -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -Xptxas -v
CSRC := spf_b200/csrc
HDRS := $(CSRC)/fft16.cuh $(CSRC)/fft_consts.h $(CSRC)/team_ops.cuh $(CSRC)/kernels.cuh $(CSRC)/tables.h $(CSRC)/graph.cuh $(CSRC)/box.cuh $(CSRC)/serial.inl include/spf_b200.h

all: spf_b200/libspf_b200.so $(CSRC)/libspf_emu.so oracle

# muxgen.cpp is host-only (MUX-circuit generator); it is linked into the product library
$(CSRC)/muxgen.o: $(CSRC)/muxgen.cpp include/spf_b200.h
	$(CXX) -O2 -std=c++17 -fPIC -Wall -c -o $@ $(CSRC)/muxgen.cpp

spf_b200/libspf_b200.so: $(CSRC)/capi.cu $(CSRC)/muxgen.o $(HDRS)
	$(NVCC) $(NVFLAGS) -shared -o $@ $(CSRC)/capi.cu $(CSRC)/muxgen.o 2> $(CSRC)/ptxas.log || (cat $(CSRC)/ptxas.log; false)

$(CSRC)/libspf_emu.so: $(CSRC)/emu.cpp $(HDRS)
	$(CXX) -O2 -march=x86-64-v3 -ffp-contract=off -std=c++17 -fPIC -shared -Wall -Wno-unknown-pragmas -o $@ $(CSRC)/emu.cpp -lpthread

oracle:
	$(MAKE) -C oracle

clean:
	rm -f spf_b200/libspf_b200.so $(CSRC)/muxgen.o $(CSRC)/libspf_emu.so $(CSRC)/ptxas.log
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
