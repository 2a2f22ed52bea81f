// rsx_scatter_dispatch.cuh -- picks the scatter kernel for one pass: record size, payload lane,
// float digits, 32/64-bit offsets, rank mode, fused partition+exchange.
#pragma once

#include "rsx_scatter.cuh"
#include "rsx_scatter2.cuh"

namespace rsx {

template <int ES, int PL, int DM, typename OffT>
cudaError_t launch_scatter_t(const ScatterParams &sp, int num_sms, cudaStream_t st) {
	const bool ticket = rank_mode() == RANK_TICKET;
	if (sp.dest_base != nullptr) { // fused partition + exchange (records only)
		if constexpr (PL == 0)
			return ticket ? launch_scatter_c<ES, PL, DM, true, OffT, RANK_TICKET, FusedCfg<ES, PL>>(sp, num_sms, st)
			              : launch_scatter_c<ES, PL, DM, true, OffT, RANK_BALLOT, FusedCfg<ES, PL>>(sp, num_sms, st);
		else
			return cudaErrorInvalidValue;
	}
	if constexpr (DM == DIGIT_SPLIT) {
		return cudaErrorInvalidValue; // key-range routing exists in fused form only
	} else {
		if (ticket) { // the register-resident kernel ranks by ticket only
			if constexpr (PreferV2<ES, PL>::value)
				return launch_scatter2_c<ES, PL, DM, OffT, Cfg2<ES, PL>>(sp, num_sms, st);
			else
				return launch_scatter_c<ES, PL, DM, false, OffT, RANK_TICKET, ScatterCfg<ES, PL>>(sp, num_sms, st);
		}
		return launch_scatter_c<ES, PL, DM, false, OffT, RANK_BALLOT, ScatterCfg<ES, PL>>(sp, num_sms, st);
	}
}

template <int ES, int PL>
cudaError_t launch_scatter_pl(const ScatterParams &sp, bool is_float, bool wide, int num_sms, cudaStream_t st) {
	if (sp.nsplit != 0) { // routing by key-range splitters (multi-GPU partition): records only
		if constexpr (PL == 0)
			return wide ? launch_scatter_t<ES, PL, DIGIT_SPLIT, unsigned long long>(sp, num_sms, st)
			            : launch_scatter_t<ES, PL, DIGIT_SPLIT, uint32_t>(sp, num_sms, st);
		else
			return cudaErrorInvalidValue;
	}
	if constexpr (ES == 4 || ES == 8 || ES == 16) { // a float/double key needs >= 4 bytes (check_layout)
		if (is_float)
			return wide ? launch_scatter_t<ES, PL, DIGIT_FLOAT, unsigned long long>(sp, num_sms, st)
			            : launch_scatter_t<ES, PL, DIGIT_FLOAT, uint32_t>(sp, num_sms, st);
	}
	if (is_float)
		return cudaErrorInvalidValue;
	return wide ? launch_scatter_t<ES, PL, DIGIT_PLAIN, unsigned long long>(sp, num_sms, st)
	            : launch_scatter_t<ES, PL, DIGIT_PLAIN, uint32_t>(sp, num_sms, st);
}

template <int ES>
cudaError_t launch_scatter_es(const ScatterParams &sp, int payload_bytes, bool is_float, bool wide,
                              int num_sms, cudaStream_t st) {
	switch (payload_bytes) {
	case 0: return launch_scatter_pl<ES, 0>(sp, is_float, wide, num_sms, st);
	case 4: return launch_scatter_pl<ES, 4>(sp, is_float, wide, num_sms, st);
	case 8: return launch_scatter_pl<ES, 8>(sp, is_float, wide, num_sms, st);
	}
	return cudaErrorInvalidValue;
}

} // namespace rsx
