# Builds libmpvss_b200.so (CUDA kernels + C ABI) for sm_100a, the test-only emulator
# and the oracle's C baseline.  `python -c "import __graft_entry__ as g; g.build()"` runs this.
NVCC      ?= nvcc
CXX       ?= g++
CSRC      := mpvss_rs_b200/csrc
NVFLAGS   := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC,-O2,-pthread
LIB       := mpvss_rs_b200/libmpvss_b200.so
CU        := $(CSRC)/api.cu $(CSRC)/comm.cu $(CSRC)/modp_api.cu $(CSRC)/modp.cu $(CSRC)/ec_api.cu $(CSRC)/ec.cu $(CSRC)/hash.cu
OBJ       := $(CU:.cu=.o) $(CSRC)/sha256_ni.o
HDR       := $(wildcard $(CSRC)/*.h $(CSRC)/*.cuh) include/mpvss_b200.h

all: $(LIB) emu cppmirror

$(CSRC)/%.o: $(CSRC)/%.cu $(HDR)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(CSRC)/sha256_ni.o: $(CSRC)/sha256_ni.cpp
	$(CXX) -O2 -fPIC -msha -msse4.1 -mssse3 -c $< -o $@

$(LIB): $(OBJ)
	$(NVCC) -shared -o $@ $(OBJ) -Xcompiler -pthread -ldl

emu: tests/emu/libemu_modp.so tests/emu/libemu_ec.so tests/emu/libemu_multibox.so tests/emu/libemu_reconstruct_batch.so tests/emu/libemu_distribute_batch.so
tests/emu/libemu_%.so: tests/emu/emu_%.cpp $(HDR)
	$(CXX) -std=c++20 -O2 -DMPVSS_SIMT_EMU -shared -fPIC -pthread -o $@ $<

# the reference's protocol tests over the C++ mirror of Participant<G> (include/mpvss_b200.hpp); runs on a GPU only
cppmirror: tests/cpp/test_participant
tests/cpp/test_participant: tests/cpp/test_participant.cpp include/mpvss_b200.hpp include/mpvss_b200.h $(LIB)
	$(CXX) -std=c++17 -O1 -Wall -Wextra -Iinclude -o $@ $< -Lmpvss_rs_b200 -lmpvss_b200 -Wl,-rpath,'$$ORIGIN/../../mpvss_rs_b200'

clean:
	rm -f $(OBJ) $(LIB) tests/emu/*.so

.PHONY: all emu cppmirror clean

# The reference itself (Rust) as the oracle's anchor: builds oracle/ref_harness against /root/reference and
# regenerates tests/golden/ref_vectors.json.  Needs cargo + the crates of /root/reference/Cargo.toml;
# neither exists in the graft image (DESIGN.md section 6), so this target only reports that there.
oracle_ref:
	@if command -v cargo >/dev/null 2>&1; then \
	  cd oracle/ref_harness && cargo build --release --target-dir ../_ref && \
	  ../_ref/release/mpvss_ref_harness > ../../tests/golden/ref_vectors.json && \
	  echo "wrote tests/golden/ref_vectors.json"; \
	else echo "oracle_ref: no cargo in this image -- parity stays pinned by KATs + independent implementations"; fi
.PHONY: oracle_ref
