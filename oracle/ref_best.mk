# oracle/ref_best.mk -- TEST INFRASTRUCTURE ONLY (never linked into the product).
# The reference encoder's tools at BEST_QUALITY (ref_tools/ref_encode_best.cc, ref_reencode_best.cc): the same
# objects and flags as Makefile's ref_encode / ref_reencode, into the same git-ignored _ref/.
#   make -C oracle -f ref_best.mk ref_best
include Makefile

.PHONY: ref_best
ifneq ($(wildcard $(REF)/decoder/decoder.cc),)
ref_best: $(OUT)/ref_encode_best $(OUT)/ref_reencode_best
else
ref_best:
	@echo "reference tree not present: using prebuilt oracle/_ref (if any)"
endif

$(OUT)/ref_encode_best: ref_tools/ref_encode_best.cc ref_tools/ref_encode.cc $(ENC_OBJS) $(OUT)/libalfalfa_ref.a
	$(CXX) $(REFFLAGS) $< $(ENC_OBJS) $(OUT)/libalfalfa_ref.a -o $@

$(OUT)/ref_reencode_best: ref_tools/ref_reencode_best.cc ref_tools/ref_reencode.cc $(ENC_OBJS) $(OUT)/libalfalfa_ref.a
	$(CXX) $(REFFLAGS) $< $(ENC_OBJS) $(OUT)/libalfalfa_ref.a -o $@
