# Builds the product library (CUDA, sm_100a only) and the test-infrastructure oracle.
NVCC ?= nvcc
CXX ?= g++
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v
CSRC := ocljpegdecoder_b200/csrc
LIBDIR := ocljpegdecoder_b200/lib
BINDIR := ocljpegdecoder_b200/bin
OBJDIR := build

LIB := $(LIBDIR)/libb2j.so
OBJS := $(OBJDIR)/kernels.o $(OBJDIR)/runtime.o $(OBJDIR)/host_parse.o $(OBJDIR)/huff_lut.o
HDRS := $(wildcard $(CSRC)/*.h) include/b2j.h

all: $(LIB) $(BINDIR)/b2jdec mathcheck oracle

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; false)

$(OBJDIR)/%.o: $(CSRC)/%.cpp $(HDRS)
	@mkdir -p $(OBJDIR)
	$(CXX) -O2 -std=c++17 -fPIC -Wall -Wextra -c $< -o $@

$(LIB): $(OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS)

# stand-alone CLI with the reference's argv contract, on the decoder.h-compatible shim
$(BINDIR)/b2jdec: $(CSRC)/refshim/b2jdec_main.cpp $(CSRC)/refshim/decoder_b2j.cpp $(CSRC)/refshim/refabi.h $(LIB)
	@mkdir -p $(BINDIR)
	$(CXX) -O2 -std=c++17 -Wall -Iinclude $(CSRC)/refshim/b2jdec_main.cpp $(CSRC)/refshim/decoder_b2j.cpp \
	    -L$(LIBDIR) -lb2j -Wl,-rpath,'$$ORIGIN/../lib' -o $@

# host-side unit-check helper: the device arithmetic header + the LUT builder compiled with g++
mathcheck: tests/native/libb2jcheck.so tests/native/libb2jsync.so
# host emulation of the self-synchronising path (walk + chunk rounds of b2j_sync.h) against a table-free sequential walk
tests/native/libb2jsync.so: tests/native/synccheck.cpp $(CSRC)/b2j_sync.h $(CSRC)/huff_lut.cpp $(CSRC)/host_parse.cpp $(CSRC)/b2j_internal.h include/b2j.h
	$(CXX) -O2 -std=c++17 -fPIC -shared -Wall -I$(CSRC) -Iinclude tests/native/synccheck.cpp $(CSRC)/huff_lut.cpp $(CSRC)/host_parse.cpp -o $@
tests/native/libb2jcheck.so: tests/native/mathcheck.cpp $(CSRC)/b2j_math.h $(CSRC)/huff_lut.cpp $(CSRC)/b2j_internal.h
	$(CXX) -O2 -std=c++17 -fPIC -shared -Wall -I$(CSRC) -Iinclude tests/native/mathcheck.cpp $(CSRC)/huff_lut.cpp -o $@

oracle:
	$(MAKE) -s -C oracle all

clean:
	rm -rf $(OBJDIR) $(LIBDIR) $(BINDIR) tests/native/*.so
	$(MAKE) -s -C oracle clean

.PHONY: all oracle clean mathcheck
