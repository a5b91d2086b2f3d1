package rpk

import (
	"strconv"
	"strings"
)

// Column producers: the pod-row side of the grid.  Restated here (not imported from the reference, which
// keeps them unexported) so that the batch path can build its columns without a *Client; semantics follow
// runpod_client.go:1102-1112 (fallback), :1115-1134 (cloud type), :1181-1191 (memory).

// AnnotationWithFallback returns the pod annotation if present and non-empty, else the owner Job's, else def.
func AnnotationWithFallback(pod, job map[string]string, key, def string) string {
	if v, ok := pod[key]; ok && v != "" {
		return v
	}
	if job != nil {
		if v, ok := job[key]; ok && v != "" {
			return v
		}
	}
	return def
}

// CloudColumn is validateCloudType folded to the engine's byte: "" and anything invalid -> SECURE.
func CloudColumn(v string) uint8 {
	switch strings.ToUpper(v) {
	case "COMMUNITY":
		return CloudCommunity
	default:
		return CloudSecure
	}
}

// ReqMemColumn is extractGPUMemory saturated to the engine's int32 column.
func ReqMemColumn(v string) int32 {
	mem := 16
	if v != "" {
		if m, err := strconv.Atoi(v); err == nil {
			mem = m
		}
	}
	if mem > 1<<31-1 {
		return 1<<31 - 1
	}
	if mem < -(1 << 31) {
		return -(1 << 31)
	}
	return int32(mem)
}

// GpuTypeIDs parses runpod.io/gpu-type-ids exactly like runpod.io/datacenter-ids (runpod_client.go:1354-1362):
// strings.Split on "," then strings.TrimSpace per element (empty elements are kept; they match no GPU type).
// "" (annotation absent, after AnnotationWithFallback) = nil: the pod is not restricted.
func GpuTypeIDs(v string) []string {
	if v == "" {
		return nil
	}
	ids := strings.Split(v, ",")
	for i, id := range ids {
		ids[i] = strings.TrimSpace(id)
	}
	return ids
}
